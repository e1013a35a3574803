"""Time the effective inflow layer (xp_effective_inflow_layer) on device-resident columns with CUDA events, in search
mode and in all-levels mode, and set it beside the per-lift yardstick -- xp_cape_cin(MU, exact_only=1), one float64
lift per column at full coalescing -- and the SB+ML+MU suite on the same columns, in the same process.

Workloads (all larger than the 126 MB L2): the ERA5 shape, 3,114,720 columns on the 37 pressure levels (float32 and
float64), and 2.8 M columns on 70 model levels (per-column pressure, float32).  Per workload and mode it prints one
JSON line: ms per call, columns/s, the gate pass fraction, the lifts and level-steps the call performs (a level-step
is one level of one lift; counted from the all-levels outputs of the same columns), level-steps/s, the lane
efficiency of the kernels' mapping (useful level-steps over 32 x the sum, over warps, of the busiest lane's), the MU
yardstick's ms and level-steps/s, the suite's ms; kernel times from torch.profiler in a pass of their own; the GPU
name and power limit.  A 5,000-column sample of each workload is checked against tests/effective_oracle.py.

    python tools/bench_effective.py [--reps 10] [--warmup 3] [--sample 5000] [--out profiles/r4_bench_effective.jsonl]
"""
import argparse
import heapq
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_downdraft import gpu_info, kernel_times, timed  # noqa: E402
from xarray_parcel_b200 import _lib, synth  # noqa: E402

# resident lanes of the layer kernel's persistent grid: 148 SMs x 3 CTAs of 128 (160-168 registers, DESIGN.md 3.13)
LAYER_LANES = 148 * 3 * 128


def work_counts(p, t, td, r_all, mu):
    """Per column [N] (torch, on the device): level-steps of the gate lift, of the search-mode layer lifts and of the
    all-levels lifts, and their lift counts.  The lift from level k covers the L - k levels with p <= p_k."""
    L, N = t.shape
    pp = p[:, None].expand(L, N) if p.dim() == 1 else p
    valid = ~(torch.isnan(pp) | torch.isnan(t) | torch.isnan(td))
    steps_k = (L - torch.arange(L, device=t.device, dtype=torch.int64))[:, None]
    ok = valid & (r_all["level_parcel_cape"] >= 100.0) & (r_all["level_parcel_cin"] > -250.0)
    k_mu = mu["level_shift"].long()
    gate = (mu["cape"] >= 100.0) & (mu["cin"] > -250.0)
    gate_steps = torch.where(k_mu < L, L - k_mu, torch.zeros_like(k_mu))
    # search: valid levels from the surface up to and including the first valid failing level above the base
    lev = torch.arange(L, device=t.device)[:, None]
    has_base = ok.any(0)
    base = torch.where(has_base, ok.to(torch.int8).argmax(0), torch.full((N,), L, device=t.device))
    fail_above = valid & ~ok & (lev > base[None, :])
    first_fail = torch.where(fail_above.any(0), fail_above.to(torch.int8).argmax(0), torch.full((N,), L, device=t.device))
    lifted = valid & (lev <= first_fail[None, :]) & (lev != k_mu[None, :]) & gate[None, :]
    search_steps = (lifted * steps_k).sum(0)
    return {"gate": gate, "gate_steps": gate_steps, "search_steps": search_steps, "search_lifts": lifted.sum(0),
            "all_steps": (valid * steps_k).sum(0), "all_lifts": valid.sum(0), "any_valid": valid.any(0)}


def static_lane_efficiency(w):
    """Adjacent columns in a warp, each lane one column: sum / (32 x sum over warps of the largest)."""
    w = w.double()
    pad = (-w.numel()) % 32
    w = torch.cat([w, torch.zeros(pad, dtype=w.dtype, device=w.device)]).view(-1, 32)
    return float(w.sum() / (32 * w.max(1).values.sum()))


def dynamic_lane_efficiency(w, lanes=LAYER_LANES):
    """The layer kernel's mapping: every lane takes the next list item when it finishes its last one (all lanes
    progressing one level-step per step).  Warp time = its busiest lane's total."""
    w = w.cpu().numpy().astype(np.int64)
    if w.size == 0:
        return None
    lanes = min(lanes, w.size)
    load = np.zeros(lanes, dtype=np.int64)
    heap = [(0, i) for i in range(lanes)]
    for x in w:
        t, i = heapq.heappop(heap)
        load[i] = t + x
        heapq.heappush(heap, (load[i], i))
    pad = (-lanes) % 32
    load = np.concatenate([load, np.zeros(pad, dtype=np.int64)]).reshape(-1, 32)
    return float(w.sum() / (32 * load.max(1).sum()))


def check_sample(ctx, p, t, td, n_sample, seed):
    import effective_oracle as eo
    from oracle import parcel as op
    from oracle import tables as otab
    N = t.shape[1]
    g = torch.Generator(device="cpu").manual_seed(seed)
    cols = torch.randperm(N, generator=g)[:n_sample].sort().values.to(t.device)
    ps = p if p.dim() == 1 else p[:, cols]
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in
           ctx.effective_inflow_layer(ps, t[:, cols], td[:, cols], profile=True).items()}
    srch = {k: v.cpu().numpy().astype(np.float64) for k, v in ctx.effective_inflow_layer(ps, t[:, cols], td[:, cols]).items()}
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    opts = op.Options(op.MoistLapseLUT(otab.AdiabatTables(pl, tl, idx, cur)))
    P, T, D = [x.cpu().numpy().astype(np.float64) for x in (ps, t[:, cols], td[:, cols])]
    ora = eo.effective_inflow_layer(P, T, D, opts)
    f32 = t.dtype == torch.float32
    cast = (lambda v: v.astype(np.float32).astype(np.float64)) if f32 else (lambda v: v)
    valid = eo.valid_levels(P, T, D)
    excuse = valid & (T == D)
    worst = 0.0
    for k in _lib.EFFECTIVE_LEVEL_FIELDS:
        y = cast(ora[k])
        assert np.array_equal(np.isnan(got[k]), np.isnan(y)), k
        with np.errstate(invalid="ignore"):
            err = np.where(np.isnan(y) | excuse, 0.0, np.abs(got[k] - y) / np.maximum(np.abs(y), 1.0))
        worst = max(worst, float(err.max()))
    assert worst <= (2.4e-7 if f32 else 1e-9), worst
    with np.errstate(invalid="ignore"):
        tol = np.maximum(np.abs(ora["level_parcel_cape"]), 1.0) * 1e-6
        near = (np.abs(ora["level_parcel_cape"] - 100.0) < tol) | (np.abs(ora["level_parcel_cin"] + 250.0) < tol)
    loose = (near | excuse).any(axis=0)
    differ = 0
    for k in _lib.EFFECTIVE_FIELDS:
        assert np.array_equal(srch[k], got[k], equal_nan=True), k
        same = np.isclose(got[k], cast(ora[k]), rtol=0, atol=0, equal_nan=True)
        assert (same | loose).all(), k
        differ += int((~same).sum())
    return {"oracle_sample_columns": n_sample, "oracle_level_max_rel_err": worst,
            "oracle_excused_columns": int(loose.sum()), "oracle_base_top_differences_in_excused": differ,
            "oracle_check": "pass"}


def run(ctx, name, p, t, td, args):
    N, L = t.shape[1], t.shape[0]
    search = lambda: ctx.effective_inflow_layer(p, t, td)                          # noqa: E731
    all_levels = lambda: ctx.effective_inflow_layer(p, t, td, profile=True)        # noqa: E731
    mu_opts = _lib.make_options(exact_only=True)
    mu_outs = ctx.alloc_outputs(t, ("mu",))
    mu_call = lambda: ctx.cape_cin(p, t, td, kinds=("mu",), options=mu_opts, out=mu_outs)   # noqa: E731
    kinds = ("sb", "ml", "mu")
    s_outs = ctx.alloc_outputs(t, kinds, shift=False)
    s_opts = _lib.make_options()
    suite = lambda: ctx.cape_cin(p, t, td, kinds=kinds, options=s_opts, out=s_outs)       # noqa: E731
    ms_search = timed(search, args.reps, args.warmup)
    ms_all = timed(all_levels, max(2, args.reps // 3), 1)
    ms_mu = timed(mu_call, args.reps, args.warmup)
    ms_suite = timed(suite, args.reps, args.warmup)
    r_all = all_levels()
    mu = mu_call()["mu"]
    w = work_counts(p, t, td, r_all, mu)
    del r_all
    gate_steps = int(w["gate_steps"].sum())
    search_steps = int(w["search_steps"].sum())
    all_steps = int(w["all_steps"].sum())
    passing = w["gate"]
    listed_all = w["all_steps"][w["any_valid"]]
    base = {"workload": name, "columns": N, "levels": L, "dtype": str(t.dtype).replace("torch.", ""),
            "pressure": "shared 1-D axis" if p.dim() == 1 else "per column",
            "gate_pass_fraction": round(float(passing.double().mean()), 4),
            "mu_exact_ms": round(ms_mu, 4), "mu_exact_level_steps_per_s": round(gate_steps / (ms_mu * 1e-3), 1),
            "suite_sb_ml_mu_ms": round(ms_suite, 4)}
    rows = []
    rows.append(dict(base, mode="search", ms=round(ms_search, 4), columns_per_s=round(N / (ms_search * 1e-3), 1),
                     lifts=int(N + w["search_lifts"].sum()), level_steps=gate_steps + search_steps,
                     lifts_per_passing_column=round(float((w["search_lifts"][passing] + 1).double().mean()), 3),
                     level_steps_per_s=round((gate_steps + search_steps) / (ms_search * 1e-3), 1),
                     lane_efficiency_gate_kernel=round(static_lane_efficiency(w["gate_steps"]), 4),
                     lane_efficiency_layer_kernel=round(dynamic_lane_efficiency(w["search_steps"][passing]), 4),
                     lane_efficiency_one_thread_per_column=round(
                         static_lane_efficiency(w["gate_steps"] + w["search_steps"]), 4),
                     ms_over_mu_exact=round(ms_search / ms_mu, 3)))
    rows.append(dict(base, mode="all_levels", ms=round(ms_all, 4), columns_per_s=round(N / (ms_all * 1e-3), 1),
                     lifts=int(w["all_lifts"].sum()), level_steps=all_steps,
                     level_steps_per_s=round(all_steps / (ms_all * 1e-3), 1),
                     lane_efficiency_layer_kernel=round(dynamic_lane_efficiency(listed_all), 4),
                     ms_over_mu_exact=round(ms_all / ms_mu, 3)))
    rows[0]["kernels"] = kernel_times([search, mu_call], reps=3)
    rows[1]["kernels"] = kernel_times([all_levels], reps=1)
    del mu_outs, s_outs
    chk = check_sample(ctx, p, t, td, min(args.sample, N), seed=7)
    for r in rows:
        r.update(chk)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=5000)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_effective.py needs a CUDA device")
    f = open(args.out, "a") if args.out else None

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        if f:
            f.write(s + "\n")
            f.flush()

    emit(gpu_info())
    ctx = _lib.get_context(0)
    ctx.tables_build()
    p, t, td = synth.era5_columns(3_114_720, seed=1234, device="cuda")
    for r in run(ctx, "era5_3114720x37_f32", p, t, td, args):
        emit(r)
    for r in run(ctx, "era5_3114720x37_f64", p.double(), t.double(), td.double(), args):
        emit(r)
    del p, t, td
    p, t, td = synth.model_level_columns(2_800_000, 70, seed=1234, device="cuda")
    for r in run(ctx, "model_2800000x70_f32", p, t, td, args):
        emit(r)
    emit(gpu_info())


if __name__ == "__main__":
    main()
