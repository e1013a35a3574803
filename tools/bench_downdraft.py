"""Time downdraft CAPE (xp_downdraft_cape) on device-resident columns with CUDA events and set it beside the SB+ML+MU
suite (xp_suite through Context.cape_cin) on the same columns, in the same process.

Workloads (both larger than the 126 MB L2): the ERA5 shape, 3,114,720 columns on the 37 pressure levels (float32 and
float64), and 2.8 M columns on 70 model levels (per-column pressure, float32).  Per workload it prints one JSON line:
ms per call, columns/s, the algorithmic bytes (the levels a column has to read, up to and including the first valid
level past 500 hPa, times the 2 or 3 input arrays, plus the three outputs) and their rate as a share of the B200's
7.7 TB/s data-sheet bandwidth and of the 6.536 TB/s copy rate measured on this project's B200; kernel times from
torch.profiler; the GPU name and power limit.  A 20,000-column sample of each workload is checked against the NumPy
oracle of tests/downdraft_oracle.py.

    python tools/bench_downdraft.py [--reps 20] [--warmup 5] [--sample 20000]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from xarray_parcel_b200 import _lib, synth  # noqa: E402

DATASHEET_TBPS = 7.7
COPY_PEAK_TBPS = 6.536      # burst device copy measured on the project's B200 (roofline.peak of profiles/r2_bench_final.json)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0]
    except Exception as e:  # the name is still reported
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def levels_read(p, t, td):
    """Levels each column must read: up to and including the first valid level below 500 hPa and not within
    np.isclose of it (all levels when there is none)."""
    L, N = t.shape
    pp = p[:, None].expand(L, N) if p.dim() == 1 else p
    valid = ~(torch.isnan(pp) | torch.isnan(t) | torch.isnan(td))
    beyond = valid & (pp.double() < 500.0 - (1e-8 + 1e-5 * 500.0))
    first = torch.where(beyond.any(0), beyond.to(torch.int8).argmax(0), torch.full((N,), L - 1, device=t.device))
    return first.to(torch.int64) + 1


def kernel_times(fns, reps=5):
    """Mean device time per launch [ms] of every kernel the callables launch, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for fn in fns:
                fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.count > 0:
            out[e.key[:120]] = {"ms_per_launch": round(t / e.count / 1000.0, 4), "launches": e.count}
    return out


def check_sample(ctx, p, t, td, n_sample, seed):
    import downdraft_oracle as dd
    from oracle import parcel as op
    from oracle import tables as otab
    N = t.shape[1]
    g = torch.Generator(device="cpu").manual_seed(seed)
    cols = torch.randperm(N, generator=g)[:n_sample].sort().values.to(t.device)
    ps = p if p.dim() == 1 else p[:, cols]
    got = ctx.downdraft_cape(ps, t[:, cols], td[:, cols], profile=True)
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    opts = op.Options(op.MoistLapseLUT(otab.AdiabatTables(pl, tl, idx, cur)))
    P, T, D = [x.cpu().numpy().astype(np.float64) for x in (ps, t[:, cols], td[:, cols])]
    ora = dd.downdraft_cape(P, T, D, opts)
    f32 = t.dtype == torch.float32
    if f32:
        ora = {k: v.astype(np.float32).astype(np.float64) for k, v in ora.items()}
    g64 = {k: v.cpu().numpy().astype(np.float64) for k, v in got.items()}
    p2 = np.broadcast_to(op._as2d(P), T.shape)
    pmax = op.nanmax(np.where(np.isnan(T) | np.isnan(D), np.nan, p2))
    ties = dd.assert_matches(g64, ora, pmax, ora["downdraft_start_pressure"], rtol=2.4e-7 if f32 else 1e-9)
    return {"oracle_sample_columns": n_sample, "oracle_tie_columns": ties, "oracle_check": "pass"}


def run(ctx, name, p, t, td, args):
    N = t.shape[1]
    elt = t.element_size()
    dd_call = lambda: ctx.downdraft_cape(p, t, td)                      # noqa: E731
    ms = timed(dd_call, args.reps, args.warmup)
    lv = levels_read(p, t, td)
    b_in = int(lv.sum().item()) * (2 if p.dim() == 1 else 3) * elt
    b_out = 3 * N * elt
    tbps = (b_in + b_out) / (ms * 1e-3) / 1e12
    kinds = ("sb", "ml", "mu")
    outs = ctx.alloc_outputs(t, kinds, shift=False)
    opts = _lib.make_options()
    suite_call = lambda: ctx.cape_cin(p, t, td, kinds=kinds, options=opts, out=outs)   # noqa: E731
    suite_ms = timed(suite_call, args.reps, args.warmup)
    res = {"workload": name, "columns": N, "levels": t.shape[0], "dtype": str(t.dtype).replace("torch.", ""),
           "pressure": "shared 1-D axis" if p.dim() == 1 else "per column",
           "dcape_ms": round(ms, 4), "dcape_columns_per_s": round(N / (ms * 1e-3), 1),
           "levels_read_mean": round(float(lv.double().mean().item()), 3),
           "algorithmic_bytes": b_in + b_out, "achieved_TBps": round(tbps, 4),
           "share_of_7.7TBps": round(tbps / DATASHEET_TBPS, 4), "share_of_6.536TBps_copy": round(tbps / COPY_PEAK_TBPS, 4),
           "suite_sb_ml_mu_ms": round(suite_ms, 4), "suite_columns_per_s": round(N / (suite_ms * 1e-3), 1),
           "dcape_over_suite_time": round(ms / suite_ms, 4)}
    res["kernels"] = kernel_times([dd_call, suite_call])
    del outs
    res.update(check_sample(ctx, p, t, td, min(args.sample, N), seed=7))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sample", type=int, default=20000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_downdraft.py needs a CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    ctx = _lib.get_context(0)
    ctx.tables_build()
    p, t, td = synth.era5_columns(3_114_720, seed=1234, device="cuda")
    print(json.dumps(run(ctx, "era5_3114720x37_f32", p, t, td, args)), flush=True)
    print(json.dumps(run(ctx, "era5_3114720x37_f64", p.double(), t.double(), td.double(), args)), flush=True)
    del p, t, td
    p, t, td = synth.model_level_columns(2_800_000, 70, seed=1234, device="cuda")
    print(json.dumps(run(ctx, "model_2800000x70_f32", p, t, td, args)), flush=True)
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
