"""Time the storm kinematics kernel (xp_storm_kinematics) and the effective-layer composition
(parcel_functions.effective_layer_parameters, split into its steps) on device-resident columns with CUDA events.

Workloads (all larger than the 126 MB L2): the ERA5 shape, 3,114,720 columns on the 37 pressure levels (float32 and
float64), and 2.8 M columns on 70 model levels (per-column pressure, float32).  Columns are tests/regime_columns.py's
real-world regimes with its seeded sheared winds and AGL heights (ERA5: "terrain" extrapolated below ground; model
levels: "synth_like"); a tenth of the columns is drawn on the host and tiled ten times on the device.

Per workload it prints one JSON line: the kinematics call as conv_properties(kinematics=True) makes it (Bunkers motion,
SRH 0-1 and 0-3 km) -- ms per call, columns/s, the algorithmic bytes (per column the levels up to the first profile
point at or above 6 km x 3 fields, the surface wind and 8 outputs) and their rate against the 7.7 TB/s data-sheet
figure; the effective composition's steps (effective inflow layer, the ML+MU lift, the four height interpolations, the
kinematics and composite kernels) in ms; kernel times from torch.profiler in a pass of their own; a 2,000-column sample
checked against tests/kinematics_oracle.py; the GPU name, power limit and max SM clock.

    python tools/bench_kinematics.py [--reps 20] [--warmup 3] [--out profiles/r5_bench_kinematics.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_downdraft import DATASHEET_TBPS, gpu_info, kernel_times, timed  # noqa: E402
from xarray_parcel_b200 import _lib  # noqa: E402
import regime_columns as rc  # noqa: E402

TILE = 10


def workload(layout, regime, n, levels, seed):
    """Device tensors p ([L] or [L, N]), T, Td, height AGL, u, v [L, N] and the surface wind [N], float32."""
    m = n // TILE
    p, t, td, p0 = rc.columns(regime, m, seed=seed, layout=layout, levels=levels)
    f = rc.conv_fields(p, t, td, p0, seed=seed + 1)
    tile = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().repeat(*([1] * (a.ndim - 1) + [TILE]))  # noqa
    dev = {"p": torch.from_numpy(p).cuda() if p.ndim == 1 else tile(p), "t": tile(f["temperature"]), "td": tile(td)}
    for k, name in (("z", "wind_height_above_surface"), ("u", "wind_u"), ("v", "wind_v"), ("su", "surface_wind_u"),
                    ("sv", "surface_wind_v")):
        dev[k] = tile(f[name])
    return dev


def levels_needed(z, u, v, top=6000.0):
    """Levels the kernel reads per column: up to and including the first kept level at or above ``top``."""
    L, N = z.shape
    kept = ~(torch.isnan(z) | torch.isnan(u) | torch.isnan(v)) & (z > 0)
    hit = kept & (z >= top)
    return torch.where(hit.any(0), hit.to(torch.int8).argmax(0) + 1, torch.full((N,), L, device=z.device))


def check_sample(ctx, d, n_sample, seed):
    import kinematics_oracle as ko
    N = d["u"].shape[1]
    g = torch.Generator(device="cpu").manual_seed(seed)
    cols = torch.randperm(N, generator=g)[:n_sample].sort().values.to(d["u"].device)
    args = [d[k][:, cols] for k in ("z", "u", "v")] + [d[k][cols] for k in ("su", "sv")]
    got = ctx.storm_kinematics(*args, depths=(1000.0, 3000.0))
    want, scale = ko.storm_kinematics(*[a.cpu().double().numpy() for a in args], 1, (1000.0, 3000.0))
    f32 = d["u"].dtype == torch.float32
    worst = 0.0
    for k, w in want.items():
        x = got[k].cpu().double().numpy()
        w = w.astype(np.float32).astype(np.float64) if f32 else w
        assert np.array_equal(np.isnan(x), np.isnan(w)), k
        tol = 1e-9 * scale[k] + (2.4e-7 * np.abs(np.nan_to_num(w)) if f32 else 0.0)
        err = np.where(np.isnan(w), 0.0, np.abs(x - w) / tol)
        worst = max(worst, float(err.max()))
    assert worst <= 1.0, worst
    return {"oracle_sample_columns": n_sample, "oracle_worst_error_over_tolerance": round(worst, 4),
            "oracle_check": "pass"}


def run(ctx, name, d, args):
    z, u, v, su, sv = d["z"], d["u"], d["v"], d["su"], d["sv"]
    p, t, td = d["p"], d["t"], d["td"]
    L, N = u.shape
    es = u.element_size()
    kin = lambda: ctx.storm_kinematics(z, u, v, su, sv, depths=(1000.0, 3000.0))        # noqa: E731
    ms_kin = timed(kin, args.reps, args.warmup)
    lev = levels_needed(z, u, v)
    nbytes = int(lev.sum()) * 3 * es + N * (2 + 8) * es
    row = {"workload": name, "columns": N, "levels": L, "dtype": str(u.dtype).replace("torch.", ""),
           "kinematics_call": "Bunkers motion + SRH 0-1, 0-3 km", "kinematics_ms": round(ms_kin, 4),
           "kinematics_columns_per_s": round(N / (ms_kin * 1e-3), 1),
           "mean_levels_read": round(float(lev.double().mean()), 3), "algorithmic_bytes": nbytes,
           "algorithmic_TBps": round(nbytes / (ms_kin * 1e-3) / 1e12, 3),
           "share_of_7.7TBps": round(nbytes / (ms_kin * 1e-3) / (DATASHEET_TBPS * 1e12), 4)}
    # the effective composition, step by step (parcel_functions.effective_layer_parameters)
    eff = lambda: ctx.effective_inflow_layer(p, t, td)                                    # noqa: E731
    lift_outs = ctx.alloc_outputs(t, ("ml", "mu"))
    lift = lambda: ctx.cape_cin(p, t, td, kinds=("ml", "mu"), out=lift_outs)              # noqa: E731
    e, lf = eff(), lift()
    base, top = e["effective_inflow_base"], e["effective_inflow_top"]
    el, lcl = lf["mu"]["el_pressure"], lf["ml"]["lcl_pressure"]
    zc = z.contiguous()
    interp = lambda: [ctx.interp_levels(p, [zc], x, log=True) for x in (base, top, el, lcl)]   # noqa: E731
    (zb,), (zt,), (zel,), (zl,) = interp()
    zb0 = torch.clamp(zb, min=0.0)
    mid = zb0 + (zel - zb0) / 2.0
    layer_kin = lambda: ctx.storm_kinematics(z, u, v, su, sv, srh_layer=(zb, zt), bwd_layer=(zb0, mid),     # noqa
                                             outputs=["srh_layer", "bulk_wind_difference"])
    r = layer_kin()
    comp = lambda: ctx.supercell_tornado_parameters(lf["mu"]["cape"], torch.nan_to_num(r["srh_layer"]),   # noqa
                                                    torch.nan_to_num(r["bulk_wind_difference"]), lf["ml"]["cape"],
                                                    lf["ml"]["cin"], zl)
    steps = {"effective_inflow_layer_ms": timed(eff, max(3, args.reps // 4), 1),
             "ml_mu_lift_ms": timed(lift, args.reps, args.warmup),
             "height_interpolations_ms": timed(interp, args.reps, args.warmup),
             "layer_kinematics_kernel_ms": timed(layer_kin, args.reps, args.warmup),
             "composite_kernel_ms": timed(comp, args.reps, args.warmup)}
    row.update({k: round(x, 4) for k, x in steps.items()})
    total = sum(steps.values())
    row["effective_composition_ms"] = round(total, 4)
    row["new_kernels_share_of_composition"] = round(
        (steps["layer_kinematics_kernel_ms"] + steps["composite_kernel_ms"]) / total, 4)
    row["gate_pass_fraction"] = round(float((~torch.isnan(base)).double().mean()), 4)
    row["kernels"] = kernel_times([kin, layer_kin, comp], reps=3)
    row.update(check_sample(ctx, d, 2000, seed=7))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_kinematics.py needs a CUDA device")
    assert args.reps >= 20, "at least 20 timed calls"
    f = open(args.out, "a") if args.out else None

    def emit(x):
        s = json.dumps(x)
        print(s, flush=True)
        if f:
            f.write(s + "\n")
            f.flush()

    emit(gpu_info())
    ctx = _lib.get_context(0)
    ctx.tables_build()
    d = workload("era5", "terrain", 3_114_720, 37, seed=1234)
    emit(run(ctx, "era5_3114720x37_f32", d, args))
    emit(run(ctx, "era5_3114720x37_f64", {k: x.double() for k, x in d.items()}, args))
    del d
    torch.cuda.empty_cache()
    d = workload("model", "synth_like", 2_800_000, 70, seed=1234)
    emit(run(ctx, "model_2800000x70_f32", d, args))
    emit(gpu_info())


if __name__ == "__main__":
    main()
