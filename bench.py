#!/usr/bin/env python
"""bench.py -- smooth Cooper-Frye spectra throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4ce] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one pass of the hot path (prepare + spectra kernel + chunk reduction [+ all-reduce]) over the whole synthetic
surface.  The default workload is BASELINE.json configs[2]: 1 000 000-cell 3+1D viscous surface, full PDG (305 species,
hrg_eos = 1), 14-moment delta-f, 32 x 24 x 21 momentum bins = 4.92e12 evaluations per step.  For N > 1 the SAME surface is
sharded by cell over the ranks (strong scaling, as north_star defines it) and the 39 MB spectra array is all-reduced (NCCL).

value  : evaluations/s with the surface already resident in HBM (CUDA events around K steps, max over ranks).
e2e    : the same metric through the C ABI with HOST buffers: H2D of the (pinned) surface arrays and D2H of the spectra
         inside the timed region.
roofline: FP64 pipe.  achieved = 85 flop/evaluation (SURVEY 8d: the reference's inner loop as written) x evaluations per
         launch / mean spectra-kernel time (CUDA events inside the C ABI, on the launch stream); peak = FP64 DFMA roof
         measured live on this GPU (MEASURED_PEAKS.json has no FP64 entry).  HBM traffic is reported to show it is not the bound.
cpu_baseline: the UNMODIFIED reference (oracle/_ref/is3d_ref_omp, -O3 -fopenmp, all host cores) on a bounded sample.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_EVAL = {1: 85.0, 2: 87.0, 3: 140.0, 4: 140.0, 5: 94.0}     # SURVEY.md section 8(d); 5 = anisotropic PL kernel
IDEAL_FLOPS = 29.0

WORKLOADS = {
    # name: (cells, dimension, df_mode, chosen, viscous, description)
    "cfg3": (1_000_000, 3, 1, "chosen_urqmd", True, "cfg3: 1M-cell 3+1D viscous surface, full PDG (305 species), 14-moment df"),
    "cfg4ce": (1_000_000, 3, 2, "chosen_urqmd", True, "cfg4: 1M-cell 3+1D viscous surface, full PDG, Chapman-Enskog df"),
    "cfg4mike": (1_000_000, 3, 3, "chosen_urqmd", True, "cfg4: 1M-cell 3+1D viscous surface, full PDG, feqmod (Mike)"),
    "cfg4jonah": (1_000_000, 3, 4, "chosen_urqmd", True, "cfg4: 1M-cell 3+1D viscous surface, full PDG, feqmod (Jonah)"),
    "cfg5": (1_000_000, 3, 5, "chosen_urqmd", True, "cfg5: 1M-cell 3+1D anisotropic-hydro surface (PL matching), full PDG, residual 14-moment df"),
    "cfg2": (100_000, 2, 1, "chosen_pikp", False, "cfg2: 100k-cell boost-invariant surface, pi/K/p, ideal f_eq, 241-point eta quadrature"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--operation", type=int, default=1, choices=[0, 1],
                    help="1: momentum spectra (headline); 0: spacetime distributions of the same integrand (SURVEY 8f N2), df_mode 1-4 workloads")
    ap.add_argument("--cells", type=int, default=0, help="override the cell count (development only; reported in config)")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--chunks", type=int, default=0, help="cell chunks per launch (0 = library default; 1 makes every block stream the whole surface)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--single-process", action="store_true",
                    help="--gpus N > 1 without torchrun: ONE process drives N GPUs through is3d_b200_smooth_spectra_multi "
                         "(cells sharded and all-reduced inside the C ABI, host arrays in and out)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64), so that two "
                         "builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm only times a CPU sample")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """arrays: {name: array} as the timed call returned them (the spectra are flat [y][phi][pT][species], 39 MB for 305 species)."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.path = tempfile.mktemp(prefix="is3d_clk_")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [[c.strip() for c in l.split(",")] for l in open(self.path).read().strip().splitlines() if l.strip()]
            sm = [float(r[0]) for r in rows]
            busy = [s for s, r in zip(sm, rows) if float(r[2]) > 250.0] or sm      # samples under load
            out["sm_mhz"] = statistics.median(busy)
            out["sm_max_mhz"] = float(rows[0][1])
            out["power_w_max"] = max(float(r[2]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            out["reasons"] = [n for j, n in enumerate(names) if any(r[3 + j].lower().startswith("active") for r in rows)]
            out["samples"] = len(rows)
        except Exception as e:          # never let monitoring break the measurement
            out["error"] = str(e)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
SPACETIME_BINS = dict(tau_min=0.0, tau_max=12.0, tau_bins=120, r_min=0.0, r_max=12.0, r_bins=60)      # iS3D_parameters.dat:82-89


def reference_sample(workload, cells=4000, n_species=4, threads=None, repeats=1, operation=1):
    """Time the unmodified reference (OpenMP build, all host cores) on a bounded sample of the workload.

    Returns dict(value evals/s, cores, kind, sample, seconds list).  Falls back to the C oracle ("port") if the reference
    binary is not present in oracle/_ref."""
    from is3d_b200 import synthetic, tables, workdir
    from oracle import cf_oracle as cfo
    n_full, dim, dfm, chosen, viscous, desc = WORKLOADS[workload]
    fx = tables.load_fixture()
    threads = threads or os.cpu_count() or 1
    if dim == 2:
        cells = max(cells // 20, 50)
    if operation == 0:
        cells = max(cells // 4, 20)                # calculate_dN_dX has no OpenMP pragma: one core whatever OMP_NUM_THREADS says
    cols = synthetic.surface_vh(cells, synthetic.SEEDS["cfg3" if dim == 3 else "cfg2"], three_d=(dim == 3), viscous=viscous)
    ids = list(fx[chosen][:n_species])
    sp = tables.species(fx, 1, ids); g = tables.grid(fx)
    evals = cells * len(ids) * len(g["pT"]) * len(g["phi"]) * (len(g["y"]) if dim == 3 else len(g["eta"]))
    secs = []
    exe = cfo.ref_binary(omp=True)
    if exe is not None:
        wd = tempfile.mkdtemp(prefix="is3d_ref_")
        try:
            workdir.materialize(wd, surface_columns=cols, chosen=ids, fixture=fx, operation=operation, mode=1, hrg_eos=1, dimension=dim,
                                df_mode=dfm, include_bulk_deltaf=int(viscous), include_shear_deltaf=int(viscous), **SPACETIME_BINS)
            for _ in range(repeats):
                _, info = cfo.run_reference(wd, what="kernel" if operation == 1 else "full", omp=True, threads=threads)
                secs.append(info["seconds"])
        finally:
            shutil.rmtree(wd, ignore_errors=True)
        kind = "reference"
        note = "unmodified reference src/cpp, g++ -O3 -fopenmp (CMakeLists.txt:11), OMP_NUM_THREADS=%d, kernel call only" % threads
        if operation == 0:
            note = "unmodified reference src/cpp, g++ -O3 -fopenmp, calculate_spectra() with operation = 0 incl. its file writers; " \
                   "calculate_dN_dX has no OpenMP pragma, so it runs on 1 core"
            threads = 1
        elif dim == 3:
            note += "; timing only: the reference's 3+1D OpenMP results are wrong (data race, SURVEY R3)"
    else:
        cells_soa = synthetic.columns_to_cells(cols, 1)
        tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
        fl = tables.flags(df_mode=dfm, dimension=dim, include_bulk=int(viscous), include_shear=int(viscous))
        os.environ["OMP_NUM_THREADS"] = str(threads)
        for _ in range(repeats):
            t0 = time.perf_counter()
            if operation == 0:
                cfo.spacetime(fl, cells_soa, sp, g, tab, SPACETIME_BINS, gla)
            else:
                cfo.smooth(fl, cells_soa, sp, g, tab, gla)
            secs.append(time.perf_counter() - t0)
        kind = "port"
        note = "oracle/cf_oracle.c (OpenMP over species, %d threads)" % threads
    best = min(secs)
    return dict(value=evals / best, unit="evaluations/s", cores=threads, kind=kind,
                sample="%d-cell prefix x first %d species of %s (%d evaluations); %s" % (cells, len(ids), chosen, evals, note),
                seconds=secs, evaluations=evals)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_full, dim, dfm, chosen, viscous, desc = WORKLOADS[args.workload]
    total = args.steps + args.warmup
    t0 = time.perf_counter()
    res = reference_sample(args.workload, repeats=total, operation=args.operation)
    if args.operation == 0:
        desc += "; operation = 0: spacetime distributions (120 tau x 60 r bins)"
    secs = res["seconds"][args.warmup:]
    mean = sum(secs) / len(secs)
    value = res["evaluations"] / mean
    line = {
        "impl": "reference", "metric": "Cooper-Frye cell*momentum*species evaluations/s", "value": value, "unit": "evaluations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "sample": res["sample"], "wall_s": time.perf_counter() - t0},
        "cpu_baseline": {"value": value, "unit": "evaluations/s", "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
        "e2e": {"value": value, "unit": "evaluations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)



# ------------------------------------------------------------------------------------------------ roofline helpers
# FP64-pipe instructions executed per evaluation (warp instructions per warp-evaluation, dead evaluations included), from the
# committed ncu captures of the default kernel of each model (profiles/README.md names the file behind every number)
FP64_INSTR_PER_EVAL = {1: 13.75,          # profiles/r2_ncu_full_shift_default.json (cf_shift_kernel; cf_kernel: 17.78, r2_ncu_full_lin14_200k_1chunk.json)
                       2: 16.11,          # profiles/r2_instr_cfg4ce_shift.csv (smsp__inst_executed_pipe_fp64.sum x 32 / evaluations; cf_kernel: 20.12)
                       3: 22.6,           # profiles/r1_ncu_full_cf_kernel_feqmod.json (Mike)
                       4: 22.69,          # profiles/r2_ncu_full_cfg4jonah.json
                       5: 27.24,          # profiles/r2_ncu_full_cfg5_vah.json
                       "ideal2d": 10.57}  # profiles/r2_ncu_full_cfg2_ideal2d.json


def alive_fraction(cells, sp, g, dim, n_sample=256, vah=False):
    """Fraction of the evaluations whose exp(u.p / T) stays finite in the reference (the others are exactly 0 there and are skipped
    by the kernels), counted on a random sample of cells with torch on the GPU: x = (p.u) / T <= ln(DBL_MAX)."""
    import torch
    n = len(cells["tau"])
    idx = np.random.default_rng(7).choice(n, size=min(n_sample, n), replace=False)
    dev = "cuda"
    t = lambda k: torch.from_numpy(np.ascontiguousarray(np.asarray(cells[k])[idx])).to(dev)
    tau, eta, ux, uy, un = t("tau"), t("eta"), t("ux"), t("uy"), t("un")
    T = t("Lambda") if vah else t("T")
    ut = torch.sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un)
    mass = torch.from_numpy(np.asarray(sp["mass"])).to(dev); pT = torch.from_numpy(np.asarray(g["pT"])).to(dev)
    phi = torch.from_numpy(np.asarray(g["phi"])).to(dev)
    if dim == 3:
        yv = torch.from_numpy(np.asarray(g["y"])).to(dev)
        d = yv[None, :] - eta[:, None]
    else:
        d = -torch.from_numpy(np.asarray(g["eta"])).to(dev)[None, :].expand(len(idx), -1)
    A = (torch.cosh(d) * ut[:, None] - tau[:, None] * torch.sinh(d) * un[:, None]) / T[:, None]          # [cell, slot]
    B = (torch.cos(phi)[None, :] * ux[:, None] + torch.sin(phi)[None, :] * uy[:, None]) / T[:, None]      # [cell, phi]
    mT = torch.sqrt(mass[:, None] ** 2 + pT[None, :] ** 2)                                               # [species, pT]
    alive = 0; total = 0
    for c0 in range(0, len(idx), 8):
        a = A[c0:c0 + 8, None, None, :, None] * mT[None, :, :, None, None]                                # cell, species, pT, slot, phi
        x = a - (pT[None, None, :, None, None] * B[c0:c0 + 8, None, None, None, :])
        alive += int((x <= 709.782712893384).sum().item()); total += x.numel()
    return alive / total


def _measured_traffic(workload, operation):
    """dram__bytes_read + dram__bytes_write of one full-size launch of the dominant kernel (ncu --set full), if a capture of this
    workload is committed under profiles/ (r2_traffic.json: {workload: bytes})."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        return d.get("%s_op%d" % (workload, operation))
    except Exception:
        return None


def run_single_process(args):
    """--gpus N --single-process: ONE process, N GPUs, through is3d_b200_smooth_spectra_multi (host arrays; cells sharded by the C
    ABI over one host thread + stream per device, one ncclAllReduce of the spectra).  Every number is end to end by construction."""
    import torch
    from is3d_b200 import api, synthetic, tables
    n_full, dim, dfm, chosen, viscous, desc = WORKLOADS[args.workload]
    if dfm == 5 or args.operation == 0:
        raise SystemExit("--single-process covers the operation = 1 viscous-hydro workloads")
    n_cells = args.cells or n_full
    n_dev = api.init_devices(args.gpus)
    if n_dev != args.gpus:
        raise SystemExit("asked for %d GPUs, library initialised %d" % (args.gpus, n_dev))
    fx = tables.load_fixture()
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx); tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    fl = tables.flags(df_mode=dfm, dimension=dim, include_bulk=int(viscous), include_shear=int(viscous))
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, synthetic.SEEDS["cfg3" if dim == 3 else "cfg2"], three_d=(dim == 3), viscous=viscous), 1)
    if dfm == 4:
        pdg = tables.pdg_table(fx, 1)
        tab.update(api.jonah_tables(pdg["mass"], pdg["gspin"].astype(float), pdg["sign"].astype(float), api.surface_averages(cells)[0], gla))
    keys = ["tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "T", "P", "E", "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi"]
    host = {k: torch.from_numpy(np.ascontiguousarray(cells[k])).pin_memory().numpy() for k in keys}
    n_bins = len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * len(g["y"])
    evals_step = n_cells * len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * (len(g["y"]) if dim == 3 else len(g["eta"]))
    out = np.zeros(n_bins)

    def step():
        out[:] = 0.0
        _, st = api.smooth_spectra(fl, host, sp, g, tab, gla, out=out, tile_variant=args.variant, multi=True)
        return st

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(0)
    t0 = time.perf_counter(); sts = []
    for _ in range(args.steps):
        sts.append(step())
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"dN": out})
    # the same surface on one device of the same process: bin-by-bin parity of the sharded result
    single = np.zeros(n_bins)
    api.smooth_spectra(fl, {k: v[:min(n_cells, 100_000)] for k, v in host.items()}, sp, g, tab, gla, out=single)
    multi_small = np.zeros(n_bins)
    api.smooth_spectra(fl, {k: v[:min(n_cells, 100_000)] for k, v in host.items()}, sp, g, tab, gla, out=multi_small, multi=True)
    nz = single != 0
    value = evals_step / (dt / args.steps)
    line = {
        "metric": "Cooper-Frye cell*momentum*species evaluations/s", "value": value, "unit": "evaluations/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "cells": n_cells, "species": len(sp["mass"]), "evaluations_per_step": evals_step,
                   "mode": "single process: is3d_b200_smooth_spectra_multi, one host thread + stream per GPU, ncclAllReduce inside the C ABI; "
                           "host arrays in, host spectra out (wall clock around the calls)",
                   "spectra_checksum": float(out.sum())},
        "clocks": clocks,
        "e2e": {"value": value, "unit": "evaluations/s", "h2d_bytes_per_step": int(len(keys) * 8 * n_cells), "d2h_bytes_per_step": int(n_bins * 8)},
        "gpu_launches": int(sum(s["gpu_launches"] for s in sts)),
        "timing": {"kernel_ms_slowest_device": float(np.mean([s["kernel_ms"] for s in sts])), "allreduce_ms": float(np.mean([s["allreduce_ms"] for s in sts])),
                   "h2d_ms": float(np.mean([s["h2d_ms"] for s in sts]))},
        "multi_gpu_parity": {"cells": int(min(n_cells, 100_000)), "max_rel_err_vs_1gpu": float(np.max(np.abs(multi_small[nz] - single[nz]) / single[nz])),
                             "zero_pattern_equal": bool(np.array_equal(single == 0, multi_small == 0))},
    }
    emit(line)

# ------------------------------------------------------------------------------------------------ our arm
# stdout carries exactly ONE line, the JSON record: while the benchmark runs, file descriptor 1 points at stderr, so that
# whatever libraries print there (NCCL's "NCCL version ..." banner when the box sets NCCL_DEBUG, the reference binary's progress
# lines) cannot precede it
_REAL_STDOUT = None


def _quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    _quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from is3d_b200 import api, distributed, synthetic, tables

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    if args.single_process:
        return run_single_process(args)
    if world > 1 or args.gpus > 1:
        if world != args.gpus:
            raise SystemExit("--gpus %d needs torchrun with %d ranks (WORLD_SIZE=%d), or --single-process" % (args.gpus, args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl")
    api.init()

    n_full, dim, dfm, chosen, viscous, desc = WORKLOADS[args.workload]
    n_cells = args.cells or n_full
    fx = tables.load_fixture()
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx); tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    vah = (dfm == 5)
    fl = tables.flags(df_mode=(1 if vah else dfm), dimension=dim, include_bulk=int(viscous), include_shear=int(viscous))
    if vah:
        fl["mode"] = 2
        cols = synthetic.surface_vah(n_cells, synthetic.SEEDS["cfg5"])
        cells = api.vah_cells(cols, fx)
    else:
        cols = synthetic.surface_vh(n_cells, synthetic.SEEDS["cfg3" if dim == 3 else "cfg2"], three_d=(dim == 3), viscous=viscous)
        cells = synthetic.columns_to_cells(cols, 1)
    del cols
    if dfm == 4:                                   # global lambda/z tables at the surface-average temperature, before sharding
        pdg = tables.pdg_table(fx, 1)
        avg = api.surface_averages(cells)
        tab.update(api.jonah_tables(pdg["mass"], pdg["gspin"].astype(float), pdg["sign"].astype(float), avg[0], gla))
    keys = ["tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "T", "P", "E", "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi"]
    spacetime = (args.operation == 0)
    if spacetime:
        if vah:
            raise SystemExit("operation = 0 has no anisotropic-hydro routine in the reference")
        keys += ["x", "y"]
        desc += "; operation = 0: spacetime distributions (120 tau x 60 r bins)"
    if vah:
        keys += ["pitt", "pitx", "pity", "pitn", "pinn", "Wx", "Wy", "Lambda", "aL", "c0", "c1", "c2", "c3", "c4"]
    lo, hi = distributed.shard_bounds(n_cells, rank, world)
    # pinned host copies of this rank's shard (e2e leg) and device-resident copies (value leg)
    host = {k: torch.from_numpy(np.ascontiguousarray(cells[k][lo:hi])).pin_memory() for k in keys}
    host_np = {k: v.numpy() for k, v in host.items()}
    dev = {k: v.cuda(non_blocking=True) for k, v in host.items()}
    del cells
    n_bins = len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * len(g["y"])
    evals_step = n_cells * len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * (len(g["y"]) if dim == 3 else len(g["eta"]))
    out = torch.zeros(n_bins, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()

    st_keys = ("dN_tau", "dN_r", "dN_taur", "dN_dydeta", "dN_dy")
    last = {}

    def spacetime_step(cells_arg, memory):
        res, st = api.spacetime_distributions(fl, cells_arg, sp, g, tab, gla, SPACETIME_BINS, memory=memory, tile_variant=args.variant)
        flat = np.concatenate([res[k].ravel() for k in st_keys])
        if world > 1:                                  # the histograms are linear in the cells: one all-reduce of the raw sums
            t = torch.from_numpy(flat).cuda()
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            flat = t.cpu().numpy()
        last["flat"] = flat; last["dN_dy"] = flat[-len(sp["mass"]):]
        last["shapes"] = [res[k].shape for k in st_keys]
        return st

    def step_outputs():
        """what a caller of the timed call receives from the last step: the spectra, or the (all-reduced) histograms"""
        if not spacetime:
            return {"dN": out.cpu().numpy()}
        sizes = [int(np.prod(s)) for s in last["shapes"]]
        parts = np.split(last["flat"], np.cumsum(sizes)[:-1])
        return {k: p.reshape(s) for k, p, s in zip(st_keys, parts, last["shapes"])}

    def step_device():
        if spacetime:
            return spacetime_step(dev, "device")
        out.zero_()
        _, st = api.smooth_spectra(fl, dev, sp, g, tab, gla, out=out, memory="device", tile_variant=args.variant, n_chunks=args.chunks)
        if world > 1:
            dist.all_reduce(out, op=dist.ReduceOp.SUM)
        return st

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # roofline denominator, measured live on this GPU before the timed region
    peak_burst, _ = api.measure_fp64_peak()
    peak_sustained = api.measure_fp64_sustained(2.0)

    for _ in range(args.warmup):
        step_device()
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    kernel_ms, prepare_ms, reduce_ms, launches = [], [], [], 0
    e0.record(stream)
    for _ in range(args.steps):
        st = step_device()
        kernel_ms.append(st["kernel_ms"]); prepare_ms.append(st["prepare_ms"]); reduce_ms.append(st["reduce_ms"])
        launches += st["gpu_launches"] + 1                     # + out.zero_() fill kernel
    e1.record(stream)
    sync_all()
    clocks = sampler.stop() if sampler else None
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:                # before the untimed repetitions and the e2e leg below recompute them
        dump_outputs(args.dump_outputs, step_outputs())
    if sampler and world == 1 and clocks.get("sm_mhz") is None:
        # the timed region is shorter than nvidia-smi's sampling period (cfg2: 57 ms per step): sample the clocks while the same
        # steps repeat, untimed, for 1.5 s
        sampler = ClockSampler(local)
        t_rep = time.perf_counter()
        while time.perf_counter() - t_rep < 1.5:
            step_device()
            torch.cuda.synchronize()
        clocks = sampler.stop()
        clocks["note"] = "sampled during an untimed 1.5 s repetition of the timed steps (timed region %.0f ms is shorter than the sampling period)" % ms_total
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        k = torch.tensor([sum(kernel_ms) / len(kernel_ms)], dtype=torch.float64, device="cuda")
        dist.all_reduce(k, op=dist.ReduceOp.MAX)
        kernel_mean = float(k.item())
    else:
        kernel_mean = sum(kernel_ms) / len(kernel_ms)
    ms_step = ms_total / args.steps
    value = evals_step / (ms_step * 1e-3)
    checksum = float(last["dN_dy"].sum()) if spacetime else float(out.sum().item())

    # ---- end to end through the C ABI with host buffers
    e2e = None
    if not args.no_e2e:
        host_out = np.zeros(n_bins)
        pinned_out = torch.zeros(n_bins, dtype=torch.float64).pin_memory()

        def step_host():
            if spacetime:                              # host arrays in, host histograms out (H2D of the shard + D2H inside the call)
                spacetime_step(host_np, "host")
                return last["dN_dy"]
            if world == 1:
                host_out[:] = 0.0
                api.smooth_spectra(fl, host_np, sp, g, tab, gla, out=host_out, tile_variant=args.variant)
                return host_out
            d = {k: v.cuda(non_blocking=True) for k, v in host.items()}       # H2D of this rank's shard, every step
            out.zero_()
            api.smooth_spectra(fl, d, sp, g, tab, gla, out=out, memory="device", tile_variant=args.variant)
            dist.all_reduce(out, op=dist.ReduceOp.SUM)
            pinned_out.copy_(out, non_blocking=False)                            # D2H of the reduced spectra
            return pinned_out.numpy()

        step_host()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = step_host()
        sync_all()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": evals_step / (dt / args.steps), "unit": "evaluations/s",
               "h2d_bytes_per_step": int(len(keys) * 8 * n_cells), "d2h_bytes_per_step": int((last["flat"].size if spacetime else n_bins) * 8 * world),
               "checksum_rel_diff": abs(float(np.sum(res)) - checksum) / abs(checksum) if checksum else 0.0}

    # ---- multi-GPU correctness inside the run (the driver's test box has one GPU): a reduced surface sharded over the ranks and
    #      all-reduced, compared bin by bin on rank 0 with the same surface computed by rank 0 alone
    multi_parity = None
    if world > 1 and not spacetime and not vah:
        n_small = 40_000
        cols_s = synthetic.surface_vh(n_small, 4321, three_d=(dim == 3), viscous=viscous)
        cells_s = synthetic.columns_to_cells(cols_s, 1)
        lo_s, hi_s = distributed.shard_bounds(n_small, rank, world)
        part = torch.zeros(n_bins, dtype=torch.float64, device="cuda")
        api.smooth_spectra(fl, {k: torch.from_numpy(np.ascontiguousarray(cells_s[k][lo_s:hi_s])).cuda() for k in keys}, sp, g, tab, gla,
                           out=part, memory="device", tile_variant=args.variant)
        dist.all_reduce(part, op=dist.ReduceOp.SUM)
        if rank == 0:
            alone = torch.zeros(n_bins, dtype=torch.float64, device="cuda")
            api.smooth_spectra(fl, {k: torch.from_numpy(np.ascontiguousarray(cells_s[k])).cuda() for k in keys}, sp, g, tab, gla,
                               out=alone, memory="device", tile_variant=args.variant)
            a = alone.cpu().numpy(); b = part.cpu().numpy(); nz = a != 0
            multi_parity = {"cells": n_small, "bins": int(a.size), "max_rel_err_vs_1gpu": float(np.max(np.abs(b[nz] - a[nz]) / np.abs(a[nz]))),
                            "zero_pattern_equal": bool(np.array_equal(a == 0, b == 0)),
                            "note": "sum of %d shard spectra (NCCL all-reduce) vs the same surface on rank 0 alone; differs by summation order only" % world}
        dist.barrier()

    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the spectra kernel) on rank 0's shard
    W = (FLOPS_PER_EVAL[dfm] if viscous else IDEAL_FLOPS)
    evals_launch = evals_step / world
    achieved = W * evals_launch / (kernel_mean * 1e-3) * 1e-12
    slots = len(g["y"]) if dim == 3 else len(g["eta"])
    rec_bytes = (hi - lo) * (slots * 48 + len(g["phi"]) * 48 + 32)         # record arrays read once per block column
    roofline = {"bound": "fp64", "achieved": achieved, "peak": peak_sustained, "unit": "TFLOP/s", "frac": achieved / peak_sustained,
                "traffic": None, "flops_per_evaluation": W, "kernel_ms": kernel_mean, "kernel_share_of_step": kernel_mean / ms_step,
                "peak_source": "measured live: dependency-free DFMA chains on all SMs, %.1f s sustained (burst %.2f TFLOP/s); "
                               "MEASURED_PEAKS.json has no FP64 entry" % (2.0, peak_burst),
                "hbm": {"record_bytes_per_launch": int(rec_bytes), "note": "algorithmic bytes = the record arrays read once + one partial "
                        "spectra array written per cell chunk; chunks are sized to a third of L2 so that the blocks sharing a chunk re-read it "
                        "from L2 (ncu at 1 M cells: 6.2 GB DRAM read + 2.3 GB written per 8.3 s launch = 1 GB/s; with 199 MB chunks the same "
                        "launch read 519 GB, profiles/r2_traffic.json): the path is not HBM-bound", "hbm_peak_gbs": _measured_hbm()},
                "reading": "W is the reference's flop count per evaluation as written (SURVEY 8d); the restructured kernel executes fewer "
                           "FP64 instructions per evaluation (fp64_instr_per_eval), so frac can exceed 1; pipe_frac is the hardware utilisation. "
                           "Issue-slot reading (profiles/r2_ubench_mix_issue.txt): on B200 a warp-wide DFMA holds the scheduler ~2 cycles and an "
                           "interleaved integer instruction ~1.7 more -- they do not overlap -- so the kernel time tracks the TOTAL warp "
                           "instruction count (30 per warp-evaluation in cf_shift_kernel, 38 in cf_kernel, at ~1.7-1.8 cycles each), not the FP64 share"}

    # hardware-side reading: FP64-pipe instructions actually executed per evaluation (ncu), the share of evaluations that are not
    # identically zero in the reference, and the resulting pipe utilisation (a warp-wide FP64 instruction holds the pipe 2 cycles)
    fkey = "ideal2d" if (dim == 2 and not viscous) else dfm
    f64i = FP64_INSTR_PER_EVAL.get(fkey)
    try:
        cells_for_alive = api.vah_cells(synthetic.surface_vah(4096, synthetic.SEEDS["cfg5"]), fx) if vah else \
            synthetic.columns_to_cells(synthetic.surface_vh(4096, synthetic.SEEDS["cfg3" if dim == 3 else "cfg2"], three_d=(dim == 3), viscous=viscous), 1)
        alive = alive_fraction(cells_for_alive, sp, g, dim, vah=vah)
    except Exception as e:
        alive = None
    evals_per_s_launch = evals_launch / (kernel_mean * 1e-3)
    roofline.update({
        "fp64_instr_per_eval": f64i,
        "pipe_frac": (f64i * evals_per_s_launch / (peak_sustained * 1e12 / 2.0)) if f64i else None,
        "alive_fraction": alive,
        "live_evaluations_per_s": (value * alive) if alive is not None else None,
        "traffic": _measured_traffic(args.workload, args.operation),
        "frac_meaning": "frac = W x evaluations/s / FP64 peak with W the REFERENCE's flop count per evaluation (SURVEY 8d): a work-normalised "
                        "speed, not a pipe utilisation; pipe_frac = executed FP64 instructions/s / (peak/2) is the hardware utilisation",
    })

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            if vah:
                raise RuntimeError("the reference cannot run this configuration: its anisotropic kernel is dead code (SURVEY R1)")
            r = reference_sample(args.workload, operation=args.operation)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:          # the baseline is a reported number, never a reason to lose the GPU measurement
            cpu = {"value": None, "unit": "evaluations/s", "cores": os.cpu_count(), "kind": "reference", "sample": "failed: %r" % (e,)}

    if spacetime:
        evals_2d = 2 if dim == 2 else 1               # 2+1D runs the integrand twice (binned yield + per-eta rapidity distribution)
        roofline["note"] = "operation = 0: same hot kernel with the momentum-integrated epilogue%s; evaluations counted once" % (
            " launched twice in 2+1D" if evals_2d == 2 else "")
    line = {
        "metric": "Cooper-Frye cell*momentum*species evaluations/s", "value": value, "unit": "evaluations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "cells": n_cells, "species": len(sp["mass"]), "momentum_bins": len(g["pT"]) * len(g["phi"]) * len(g["y"]),
                   "evaluations_per_step": evals_step, "sharding": "cells split contiguously over %d rank(s), one all-reduce of %d doubles" % (world, last["flat"].size if spacetime else n_bins),
                   "l2": "inputs larger than L2: %.0f MB of raw cell arrays + %.0f MB of per-cell records per rank vs 126 MB L2"
                         % (len(keys) * 8 * (hi - lo) / 1e6, rec_bytes / 1e6),
                   "tile_variant": args.variant, "underflow_skip": "evaluations whose exp(u.p/T) overflows (f = 0 exactly in the reference) are skipped; they still count as evaluations",
                   "spectra_checksum": checksum},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        "fraction_of_fp64_peak": achieved / peak_sustained, "multi_gpu_parity": multi_parity,
        "timing": {"prepare_ms": sum(prepare_ms) / len(prepare_ms), "kernel_ms": kernel_mean, "reduce_ms": sum(reduce_ms) / len(reduce_ms)},
    }
    emit(line)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def _measured_hbm():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6650.0          # fallback stated in B200_PROFILING.md


if __name__ == "__main__":
    main()
