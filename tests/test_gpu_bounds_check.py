"""Device-side bounds checks in place of compute-sanitizer (closed on the B200 pool, profiles/r2_sanitizer_pool_closed.txt).

``libxparcel_check.so`` (built by ``__graft_entry__.build()`` with -DXP_BOUNDS_CHECK) asserts every computed index of
the fast kernels -- shared-memory stash and coefficient table, the uncertain-column list, the 32-bit T/Td offsets --
and traps on a violation, which surfaces as a CUDA error in the child process below.  The child drives the fast
kernels over the awkward inputs: NaN-laden and all-NaN columns, saturated parcels, 3-level and 56-level axes, axes
reaching above the table top, column counts that are not a multiple of the tile, specific-humidity input; and the
regime columns of tests/regime_columns.py -- cold parcels, surfaces above 1100 hPa and model tops at 0.01 hPa (table rows
outside the segments, every column on the fix-up list: three lists of N items), ERA5 levels masked below ground.  DCAPE
and the effective inflow layer (search and all-levels mode, the gate's column list) run on regime columns too: the
staged per-column readers (40 and 16 levels), the 0.01 hPa top at 137 levels per column and on a shared axis, surfaces
above 1100 hPa and masked ERA5 levels."""

import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECK_LIB = os.path.join(ROOT, "xarray_parcel_b200", "libxparcel_check.so")

CHILD = r"""
import os, sys
sys.path.insert(0, %r)
sys.path.insert(0, os.path.join(sys.path[0], "tests"))
import numpy as np, torch
import regime_columns as rc
from xarray_parcel_b200 import _lib, synth
ctx = _lib.get_context(0)
ctx.tables_build()
def run(p, t, td, **kw):
    r = ctx.cape_cin(p.cuda(), t.cuda(), td.cuda(), kinds=("sb", "ml", "mu"), **kw)
    torch.cuda.synchronize()
    return r
n_cases = 0
for n in (1, 31, 640, 641, 100003):
    run(*synth.era5_columns(n, seed=n, nan_columns=0.05, allnan_columns=0.01, saturated=0.1)); n_cases += 1
    run(*synth.model_level_columns(n, 70, seed=n, nan_columns=0.05, allnan_columns=0.01, saturated=0.1)); n_cases += 1
# short / long / odd shared axes
for levels in ([1000, 900, 800], [1000 - 17 * k for k in range(56)], [1050, 1000, 950, 700, 400, 150, 60, 20, 4, 2.6, 2.4, 1.0]):
    L, n = len(levels), 5000
    p = torch.tensor(levels, dtype=torch.float32)
    _, t37, td37 = synth.era5_columns(n, seed=L)
    idx = torch.linspace(0, 36, L).long()
    run(p, t37[idx].contiguous(), td37[idx].contiguous()); n_cases += 1
# specific humidity in place of the dewpoint (converted in the load stage)
p, t, td = synth.era5_columns(50000, seed=5)
e = 6.112 * torch.exp(17.67 * (td - 273.15) / (td - 29.65))
w = 0.622 * e / (p[:, None] - e)
run(p, t, (w / (1 + w)).contiguous(), specific_humidity=True); n_cases += 1
# profile rows from the per-column-pressure kernel
p, t, td = synth.model_level_columns(20000, 90, seed=9)
r = ctx.cape_cin(p.cuda(), t.cuda(), td.cuda(), kinds=("mu",), profile=True); torch.cuda.synchronize(); n_cases += 1
# regime columns: the table route (three kinds), the gather route (one kind), the shared axis
for regime, kw in (("cold", {}), ("above_1100", {}), ("synth_like", dict(levels=137, p_top=0.01)),
                   ("synth_like", dict(levels=150, p_top=0.01)), ("masked", dict(layout="era5_masked"))):
    p, t, td, _ = rc.columns(regime, 3001, seed=7, **kw)
    p, t, td = (torch.from_numpy(x) for x in (p, t, td))
    run(p, t, td); n_cases += 1
    r = ctx.cape_cin(p.cuda(), t.cuda(), td.cuda(), kinds=("mu",)); torch.cuda.synchronize(); n_cases += 1
# DCAPE and the effective layer in both modes, float32 and float64
for regime, kw in (("terrain", dict(levels=40)), ("terrain", dict(levels=16)), ("synth_like", dict(levels=137, p_top=0.01)),
                   ("synth_like", dict(layout="axis", levels=137, p_top=0.01)), ("above_1100", {}),
                   ("masked", dict(layout="era5_masked"))):
    p, t, td, _ = rc.columns(regime, 3001, seed=8, **kw)
    for dt in (torch.float32, torch.float64):
        pg, tg, tdg = (torch.from_numpy(x).to(dt).cuda() for x in (p, t, td))
        ctx.downdraft_cape(pg, tg, tdg, profile=True)
        ctx.effective_inflow_layer(pg, tg, tdg)
        ctx.effective_inflow_layer(pg, tg, tdg, profile=True)
        torch.cuda.synchronize(); n_cases += 1
print("BOUNDS_CHECK_OK", n_cases)
"""


@pytest.mark.gpu
def test_fast_kernels_run_clean_with_device_bounds_checks():
    assert os.path.exists(CHECK_LIB), "run __graft_entry__.build() first (it builds the XP_BOUNDS_CHECK variant)"
    env = dict(os.environ, XP_LIB_PATH=CHECK_LIB)
    res = subprocess.run([sys.executable, "-c", CHILD % ROOT], env=env, capture_output=True, text=True, timeout=900)
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0, tail
    assert "BOUNDS_CHECK_OK" in res.stdout and "XP_BOUNDS_CHECK failed" not in tail, tail
