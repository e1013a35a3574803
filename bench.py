#!/usr/bin/env python
"""bench.py -- columns/s of the SB+ML+MU CAPE/CIN/LCL/LFC/EL suite on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the fused suite kernel over this rank's column block.  The default
workload is the ERA5-shaped configuration the metric is quoted on (BASELINE.json configs[3]:
1440 x 721 grid points x 37 pressure levels, hourly fields, full SB+ML+MU suite): every rank
holds ``--hours-per-gpu`` (default 3) hourly fields = 3.11 M columns, so 8 ranks process exactly
the named 24-hour grid per step (weak scaling: per-GPU work is fixed; columns are independent,
no collective in the data path).  Synthetic atmospheres come from xarray_parcel_b200.synth
(seeded); inputs are float32, level-major.

Prints ONE JSON line (rank 0).  ``value`` = columns/s with inputs resident in HBM (device time,
CUDA events on the launch stream, max over ranks); ``e2e`` = the same metric through the C ABI
with HOST buffers (pinned host -> device -> kernel -> host inside the timed region);
``roofline`` = algorithmic bytes / kernel time against MEASURED_PEAKS.json; ``cpu_baseline`` =
the NumPy oracle (restated reference) timed on this box's host cores on a bounded sample.
``--impl reference`` times that CPU restatement alone, with all host cores.

``--dump-outputs DIR`` writes the arrays the last timed step returned, one ``DIR/<kind>_<field>.npy`` per output, so
that two builds can be compared output for output (the inputs are seeded: the same arguments give the same inputs).
Undefined outputs (NaN: no LFC / EL) are written as 0 beside a ``DIR/<kind>_<field>_defined.npy`` mask, so every
file is finite.  Outputs larger than 60 MB in all are cut to the same seeded sample of columns in every file.

The tree is only read (it may be read-only): no bytecode is written and the oracle's tables are regenerated in memory.
"""

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "columns/sec for SB+ML+MU CAPE/CIN suite"
UNIT = "columns/s"
ERA5_NX, ERA5_NY, ERA5_NL = 1440, 721, 37
BENCH_FIELDS = {
    "sb": ["cape", "cin", "lcl_pressure", "lcl_temperature", "lcl_virtual_temperature",
           "lfc_pressure", "lfc_temperature", "el_pressure", "el_temperature"],
}
BENCH_FIELDS["ml"] = BENCH_FIELDS["sb"] + ["parcel_pressure", "parcel_temperature", "parcel_dewpoint"]
BENCH_FIELDS["mu"] = BENCH_FIELDS["ml"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="era5_suite",
                    choices=["era5_suite", "model70_sb", "model70_sb_ml", "model90_mu_profile"])
    ap.add_argument("--hours-per-gpu", type=int, default=3)
    ap.add_argument("--columns", type=int, default=0, help="override the per-GPU column count")
    ap.add_argument("--cpu-sample", type=int, default=100_000,
                    help="columns of the workload timed on the CPU oracle (0 = skip)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--ref-columns", type=int, default=0, help="--impl reference: columns per step")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra lines of the default run (other BASELINE configs, float64 I/O, pageable e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<kind>_<field>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


# ------------------------------------------------------------------------------- workloads
def workload_spec(args):
    """(name, kinds, n_levels, n_columns per GPU, pressure_is_1d, profile, description)."""
    if args.workload == "era5_suite":
        n = ERA5_NX * ERA5_NY * args.hours_per_gpu
        return dict(name=f"era5_{ERA5_NX}x{ERA5_NY}x{ERA5_NL}_x{args.hours_per_gpu}h_per_gpu_sb+ml+mu",
                    kinds=("sb", "ml", "mu"), L=ERA5_NL, N=args.columns or n, p1d=True, profile=False)
    if args.workload == "model70_sb":           # BASELINE configs[1]
        return dict(name="model_levels_1Mx70_sb", kinds=("sb",), L=70, N=args.columns or 1_000_000,
                    p1d=False, profile=False)
    if args.workload == "model70_sb_ml":        # BASELINE configs[2], one hourly step per pass
        return dict(name="aus400_2.8Mx70_sb+ml", kinds=("sb", "ml"), L=70, N=args.columns or 2_800_000,
                    p1d=False, profile=False)
    return dict(name="model_levels_10Mx90_mu_profile", kinds=("mu",), L=90,                 # configs[4]
                N=args.columns or 10_000_000, p1d=False, profile=True)


def make_inputs(spec, seed, device):
    from xarray_parcel_b200 import synth
    if spec["p1d"]:
        return synth.era5_columns(spec["N"], seed=seed, device=device)
    return synth.model_level_columns(spec["N"], spec["L"], seed=seed, device=device)


def algorithmic_bytes(spec, elt=4):
    """SURVEY.md 8(d): every input array read once, every requested output written once."""
    L, N = spec["L"], spec["N"]
    b_in = (2 if spec["p1d"] else 3) * L * elt * N + (L * elt if spec["p1d"] else 0)
    per_col_out = sum(len(BENCH_FIELDS[k]) for k in spec["kinds"]) * elt
    if spec["profile"]:
        per_col_out += 6 * (L + 1) * elt * len(spec["kinds"])
    return b_in, per_col_out * N


def config_dict(spec):
    """The `config` of the JSON line -- identical in the B200 arm and in --impl reference (same workload; the
    reference arm times a bounded SAMPLE of it per step and says so in cpu_baseline.sample)."""
    b_in, _ = algorithmic_bytes(spec)
    return {"workload": spec["name"], "columns_per_gpu": spec["N"], "levels": spec["L"],
            "parcels": list(spec["kinds"]), "io_dtype": "f32",
            "pressure": "shared 1-D axis" if spec["p1d"] else "per column",
            "profile_rows": bool(spec["profile"]),
            "l2": f"inputs {b_in / 1e6:.0f} MB per step > 126 MB L2, no flush needed",
            "sharding": "column blocks, one per GPU, no collective"}


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index, period=0.02):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for name, bit in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------- CPU oracle legs
def _oracle_chunk(job):
    """Worker: the restated reference suite on one column chunk (pressure broadcast like the
    reference's xarray broadcasting of a 1-D pressure coordinate)."""
    import numpy as np
    from oracle import parcel as op
    p, t, td = job
    if p.ndim == 1:
        p = np.broadcast_to(p[:, None], t.shape)
    opts = op.Options(op.MoistLapseLUT(_ORACLE_TABLES), lcl_mode="scipy")
    kinds = _ORACLE_KINDS
    if kinds == ("sb", "ml", "mu"):
        op.suite(p, t, td, opts)
    else:
        fns = {"sb": op.surface_based_cape_cin, "ml": op.mixed_layer_cape_cin,
               "mu": op.most_unstable_cape_cin}
        for k in kinds:
            fns[k](p, t, td, opts)
    return t.shape[1]


_ORACLE_TABLES = None
_ORACLE_KINDS = ("sb", "ml", "mu")


def oracle_setup(kinds):
    global _ORACLE_TABLES, _ORACLE_KINDS
    from oracle import tables as otab
    if _ORACLE_TABLES is None:
        _ORACLE_TABLES = otab.load_tables(cache=False)      # ~10 s; no cache file in the tree
    _ORACLE_KINDS = tuple(kinds)


def oracle_jobs(p, t, td, chunk):
    import numpy as np
    P = p.numpy().astype(np.float64)
    T = t.numpy().astype(np.float64)
    D = td.numpy().astype(np.float64)
    jobs = []
    for s in range(0, T.shape[1], chunk):
        e = min(T.shape[1], s + chunk)
        jobs.append((P if P.ndim == 1 else np.ascontiguousarray(P[:, s:e]),
                     np.ascontiguousarray(T[:, s:e]), np.ascontiguousarray(D[:, s:e])))
    return jobs


def cpu_baseline_port(spec, n_sample, seed):
    """The NumPy oracle on ONE host thread over the first ``n_sample`` columns of the workload."""
    oracle_setup(spec["kinds"])
    sub = dict(spec, N=n_sample)
    p, t, td = make_inputs(sub, seed, "cpu")
    jobs = oracle_jobs(p, t, td, 8192)
    _oracle_chunk(jobs[0])                      # warm-up (imports, caches)
    t0 = time.perf_counter()
    done = sum(_oracle_chunk(j) for j in jobs)
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"first {done} columns of the workload ({spec['name']}), NumPy float64 "
                      f"restatement of parcel_functions.py in 8192-column chunks, {dt:.1f} s"}


def run_reference(args):
    """--impl reference: the restated reference (oracle port; the xarray/MetPy original cannot be
    installed here -- DESIGN.md) on all host cores, columns chunked over a process pool like the
    reference's dask LocalCluster."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    spec = workload_spec(args)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cores = max(1, min(cores, 64))
    chunk = 4096
    n_cols = args.ref_columns or cores * chunk * 2
    oracle_setup(spec["kinds"])
    sub = dict(spec, N=n_cols)
    p, t, td = make_inputs(sub, 4321, "cpu")
    jobs = oracle_jobs(p, t, td, chunk)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(_oracle_chunk, jobs)
        t0 = time.perf_counter()
        done = 0
        for _ in range(args.steps):
            done += sum(pool.map(_oracle_chunk, jobs))
        dt = time.perf_counter() - t0
    value = done / dt
    sample = (f"{n_cols} columns per step of {spec['name']} in {chunk}-column chunks over a "
              f"{cores}-process pool, NumPy float64 restatement (oracle/), {dt:.1f} s timed")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": config_dict(spec),
            "sample_columns_per_step": n_cols,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


# ------------------------------------------------------------------------------- the B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from xarray_parcel_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    # one process per GPU: stay on the CPU cores / NUMA node next to it (the e2e path is PCIe-bound and its pinned
    # staging buffers are placed by first touch); XP_BENCH_NO_BIND=1 keeps the inherited affinity
    cpus = None
    if not os.environ.get("XP_BENCH_NO_BIND"):
        from xarray_parcel_b200.partition import bind_host_thread_to_device
        cpus = bind_host_thread_to_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    spec = workload_spec(args)
    ctx = _lib.get_context(local)
    ctx.tables_build()
    seed = 1234 + rank                                   # every rank its own columns
    p, t, td = make_inputs(spec, seed, dev)
    kinds = spec["kinds"]
    outs = ctx.alloc_outputs(t, kinds, profile=spec["profile"], fields=BENCH_FIELDS, shift=False)
    opts = _lib.make_options()
    b_in, b_out = algorithmic_bytes(spec)

    def step():
        ctx.cape_cin(p, t, td, kinds=kinds, options=opts, out=outs)

    # ---- device-resident throughput ("value") + per-launch kernel time ("roofline") ----------
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    sampler.start()
    evs[0].record()
    for i in range(args.steps):
        step()
        evs[i + 1].record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:          # before later loops reuse `outs`
        dump_outputs(args.dump_outputs, outs, spec["N"])
    total_ms = evs[0].elapsed_time(evs[-1])
    per_ms = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps))
    kernel_ms = sum(per_ms) / len(per_ms)
    launches = ctx.launch_count() - launches0
    total_ms = max_over_ranks(total_ms)
    value = spec["N"] * world * args.steps / (total_ms * 1e-3)
    flags = ctx.take_flags()
    n_exact = ctx.last_exact_count()
    # the step split at the launch of the float64 fix-up kernel (CUDA events of the library on its launch stream; a
    # separate short loop, because reading the split synchronises): the float32 sweep is the dominant kernel
    split = None
    if n_exact >= 0:
        try:
            sw, fx = [], []
            for _ in range(min(args.steps, 20)):
                step()
                a, b = ctx.last_kernel_split_ms()
                sw.append(a); fx.append(b)
            split = (sum(sw) / len(sw), sum(fx) / len(fx))
        except Exception:
            split = None

    # ---- end to end through the C ABI with host buffers --------------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    hp, ht, htd = [x.cpu().pin_memory() for x in (p, t, td)]
    houts = ctx.alloc_outputs(ht, kinds, profile=spec["profile"], pin_outputs=True,
                              fields=BENCH_FIELDS, shift=False)
    h2d = sum(x.numel() * x.element_size() for x in (hp, ht, htd))
    d2h = ctx.output_bytes(houts)
    for _ in range(2):
        ctx.cape_cin(hp, ht, htd, kinds=kinds, options=opts, out=houts)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = ctx.cape_cin(hp, ht, htd, kinds=kinds, options=opts, out=houts)   # returns when outputs are on the host
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = spec["N"] * world * e2e_steps / e2e_s
    first = kinds[0]
    e2e_check = float(torch.nan_to_num(r[first]["cape"]).double().sum())
    dev_check = float(torch.nan_to_num(outs[first][1][0]).double().sum())

    # ---- extras of the default single-GPU run: the other BASELINE configs, float64 I/O, pageable e2e ------------
    extras = None
    if rank == 0 and world == 1 and args.workload == "era5_suite" and not args.no_extras:
        extras = run_extras(args, ctx, spec, p, t, td, opts, hp, ht, htd, houts)

    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        try:
            cpu = cpu_baseline_port(spec, min(args.cpu_sample, spec["N"]), seed)
        except Exception as e:                           # the bench line must still be printed
            cpu = {"error": repr(e)}

    if rank == 0:
        peaks, peak_src = None, "fallback (B200_PROFILING.md: 6650 GB/s)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
            peak = float(peaks["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        except Exception:
            peak = 6650.0
        achieved = (b_in + b_out) / (kernel_ms * 1e-3) / 1e9
        traffic = None
        try:            # DRAM bytes of the dominant kernel from the committed ncu capture of this workload
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tr = json.load(f)
            if tr.get("workload") == spec["name"] and n_exact >= 0:
                traffic = tr["dram_bytes_per_launch"]
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if n_exact >= 0 else "f64",
            "data": "synthetic",
            "config": config_dict(spec),
            "arithmetic": ("float32 sweep + float64 LCL/mixed-layer means; columns with a decision "
                           "inside the float32 margin recomputed in float64" if n_exact >= 0 else "float64"),
            "host_cpus_rank0": (f"{len(cpus)} cores next to the GPU (NVML affinity)" if cpus else "inherited"),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "timer": "host wall clock around xp_suite(mem=HOST), max over ranks",
                    "checksum_matches_device_run": abs(e2e_check - dev_check) <= 1e-6 * max(1.0, abs(dev_check))},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": ("xp::suite_fast_kernel + prep/coef + suite_list_kernel (exact fix-up)"
                                    if n_exact >= 0 else "xp::cape_cin_kernel<float>"),
                         "kernel_ms": kernel_ms,
                         "kernel_ms_min": per_ms[0], "algorithmic_bytes_per_launch": b_in + b_out,
                         "bytes_per_column": (b_in + b_out) / spec["N"],
                         # `achieved` / `frac` above charge the WHOLE step (sweep + fix-up) to the algorithmic bytes;
                         # the sweep alone, which moves all of them, is the dominant kernel:
                         "dominant_kernel": (None if split is None else {
                             "what": "float32 sweep (axis preparation + coefficient + sweep kernels), events of the "
                                     "library around it; the float64 fix-up kernel follows",
                             "ms": split[0], "fixup_ms": split[1],
                             "achieved": (b_in + b_out) / (split[0] * 1e-3) / 1e9,
                             "frac": (b_in + b_out) / (split[0] * 1e-3) / 1e9 / peak})},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "reference_assert_flags": flags,
            "exact_path_columns": n_exact,
        }
        if extras:
            line["extras"] = extras
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 60_000_000       # --dump-outputs: under 64 MB with the .npy headers
DUMP_SEED = 20261020


def dump_outputs(out_dir, outs, n_columns):
    """Write every output block of ``ctx.alloc_outputs`` as out_dir/<kind>_<field>.npy ([N] scalars, [L+1, N]
    profile rows).  An output the library leaves undefined is NaN (no LFC / EL, all-NaN input column); the dump keeps
    every file finite: such entries are written as 0 and <kind>_<field>_defined.npy holds 1 where the value is
    defined and 0 where it is not (one for every output, so the file set does not depend on the data).  When the
    whole set exceeds DUMP_BYTES, every file holds the same sorted sample of columns drawn with DUMP_SEED, so dumps
    of two builds with the same arguments line up column for column."""
    import numpy as np
    import torch
    from xarray_parcel_b200._lib import PROFILE_FIELDS
    arrays = {}
    for kind, (_, scal, _, prof, names) in outs.items():
        for i, f in enumerate(names):
            arrays[f"{kind}_{f}"] = scal[i]
        if prof is not None:
            for i, f in enumerate(PROFILE_FIELDS):
                arrays[f"{kind}_{f}"] = prof[i]
    per_column = 2 * sum(a.numel() // n_columns * a.element_size() for a in arrays.values())    # values + masks
    n = min(n_columns, DUMP_BYTES // per_column)
    idx = None
    if n < n_columns:
        pick = np.sort(np.random.default_rng(DUMP_SEED).choice(n_columns, n, replace=False))
        idx = torch.from_numpy(pick).to(next(iter(arrays.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if idx is not None:
            a = a.index_select(a.dim() - 1, idx)
        defined = torch.isfinite(a)
        np.save(os.path.join(out_dir, name + ".npy"), torch.where(defined, a, torch.zeros_like(a)).cpu().numpy())
        np.save(os.path.join(out_dir, name + "_defined.npy"), defined.to(a.dtype).cpu().numpy())


def _time_device(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_extras(args, ctx, spec, p, t, td, opts, hp, ht, htd, houts):
    """Extra measurements of the default run (rank 0, one GPU; every one a few seconds):
      other_configs  the model-level BASELINE configs ([1] 1 M x 70 SB, [2] 2.8 M x 70 SB+ML, [4] 10 M x 90 MU + profile
                     rows): columns/s with inputs resident in HBM and the fraction of their own HBM roofline;
      f64_io         the same ERA5 suite with float64 inputs and outputs (the reference's dtype): exact float64 kernel;
      e2e_pageable   the suite through the reference-facing Python function (parcel_functions.parcel_suite) from
                     PAGEABLE NumPy arrays -- what an xarray user holds -- result Dataset on the host."""
    import numpy as np
    import torch
    out = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
    except Exception:
        peak = 6650.0
    others = {}
    for wl in ("model70_sb", "model70_sb_ml", "model90_mu_profile"):
        a2 = argparse.Namespace(**vars(args))
        a2.workload, a2.columns = wl, 0
        sp = workload_spec(a2)
        try:
            q = make_inputs(sp, 1234, p.device)
            o2 = ctx.alloc_outputs(q[1], sp["kinds"], profile=sp["profile"], fields=BENCH_FIELDS, shift=False)
            ms = _time_device(lambda: ctx.cape_cin(*q, kinds=sp["kinds"], options=opts, out=o2), 10, 3)
            bi, bo = algorithmic_bytes(sp)
            others[wl] = {"config": config_dict(sp), "value": sp["N"] / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                          "roofline_frac": (bi + bo) / (ms * 1e-3) / 1e9 / peak,
                          "bytes_per_column": (bi + bo) / sp["N"], "exact_path_columns": ctx.last_exact_count()}
            del q, o2
        except Exception as e:
            others[wl] = {"error": repr(e)}
        torch.cuda.empty_cache()
    out["other_configs"] = others
    try:                                      # float64 I/O (the reference's dtype), same columns
        n64 = spec["N"]
        p64 = p.double() if p.dim() == 1 else p.double().contiguous()
        t64, td64 = t.double().contiguous(), td.double().contiguous()
        o64 = ctx.alloc_outputs(t64, spec["kinds"], profile=False, fields=BENCH_FIELDS, shift=False)
        ms = _time_device(lambda: ctx.cape_cin(p64, t64, td64, kinds=spec["kinds"], options=opts, out=o64), 10, 3)
        fast64 = ctx.last_exact_count() >= 0
        bi, bo = algorithmic_bytes(dict(spec, N=n64), elt=8)
        out["f64_io"] = {"columns": n64, "value": n64 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                         "roofline_frac": (bi + bo) / (ms * 1e-3) / 1e9 / peak, "bytes_per_column": (bi + bo) / n64,
                         "kernel": ("xp::suite_fast_kernel<..., double> (float32 sweep of float64 columns, float64 "
                                    "parcels) + suite_list_kernel<double>" if fast64
                                    else "xp::cape_cin_kernel<double> (float64 exact path)"),
                         "exact_path_columns": ctx.last_exact_count()}
        del p64, t64, td64, o64
    except Exception as e:
        out["f64_io"] = {"error": repr(e)}
    try:                                      # pageable NumPy in, host Dataset out, through the public function
        import xarray_parcel_b200.parcel_functions as pf
        P, T, D = [np.array(x.numpy()) for x in (hp, ht, htd)]          # fresh pageable copies
        pf.parcel_suite(P, T, D, vert_axis=0)
        t0 = time.perf_counter()
        n_rep = 3
        for _ in range(n_rep):
            ds = pf.parcel_suite(P, T, D, vert_axis=0)
        dt = (time.perf_counter() - t0) / n_rep
        out["e2e_pageable"] = {"value": spec["N"] / dt, "unit": UNIT, "seconds_per_call": dt,
                               "api": "parcel_functions.parcel_suite(numpy float32 arrays, pageable) -> Dataset of "
                                      "NumPy arrays; includes the driver's staging of pageable memory and the "
                                      "allocation of the result arrays",
                               "variables": len(ds)}
    except Exception as e:
        out["e2e_pageable"] = {"error": repr(e)}
    return out


_JSON_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on
    some boxes), so keep the real stdout for the JSON line and point fd 1 at stderr for everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    sys.dont_write_bytecode = True
    _claim_stdout()
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
