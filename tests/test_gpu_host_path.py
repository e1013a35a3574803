"""The host-memory staging path (``run_host`` in xp_api.cu) block by block against the device path.

Every call with NumPy arrays or CPU tensors goes through ``run_host``: column blocks of ``XP_HOST_BLOCK_MB`` per slot,
three slot streams, page-locked mirrors that host threads fill from pageable arrays, 2-D copies with a source pitch for
blocks that are slices of wider arrays, and output copies held back until their slot is reused (``retire``) or the call
drains.  Each host call here is compared with the same call on CUDA tensors of the same arrays on the same context, so
the tables and options are identical by construction.  Columns are independent and block starts are multiples of 1024
columns, so every output must be bit-identical (compared as integer views, NaN payloads included), the reference-assert
flags must be the same, and so must ``last_exact_count``.  Contexts with 1 MB blocks make a call of a few thousand
columns run seven or more blocks; each case asserts through ``launch_count`` how many blocks actually ran.
"""

import os
from dataclasses import dataclass

import numpy as np
import pytest
import torch

import regime_columns as rc
from oracle import parcel as op
from oracle import tables as otab
from test_gpu_parity import _check
from xarray_parcel_b200 import _lib, synth

pytestmark = pytest.mark.gpu

KINDS3 = ("sb", "ml", "mu")
FORMS = ("pageable", "pinned", "pageable_slice", "pinned_slice")
DEFAULT_BLOCK_MB = 192          # xp_context::host_block_mb
SENTINEL = -7777.0              # host outputs are filled with it: a block that is never copied out shows


# --------------------------------------------------------------------------- run_host's block size
def per_column_bytes(L, es, p1d, kinds, profile=False, fields=None, shift=True):
    """Device bytes per column of one ``run_host`` call: the inputs and every requested output (xp_api.cu)."""
    n = (2 if p1d else 3) * L * es
    n_fields = len(_lib.SCALAR_FIELDS) if fields is None else len([f for f in _lib.SCALAR_FIELDS if f in fields])
    for _ in kinds:
        n += n_fields * es + (4 if shift else 0) + (len(_lib.PROFILE_FIELDS) * (L + 1) * es if profile else 0)
    if "explicit" in kinds:
        n += 3 * es
    return n


def host_blocks(n, per_col, mb):
    """(columns per block, number of blocks) of a ``run_host`` call over ``n`` columns with ``mb`` MB blocks."""
    if n == 0:
        return 0, 0
    c = max(1024, (mb << 20) // per_col // 1024 * 1024)
    c = min(c, (n + 1023) // 1024 * 1024)
    return c, -(-n // c)


# --------------------------------------------------------------------------- contexts and memory forms
@pytest.fixture(scope="module", autouse=True)
def global_context():
    """The process-wide context (``parcel_suite``, the device references) is created before any test here sets the
    staging variables, so it keeps the default block size."""
    assert "XP_HOST_BLOCK_MB" not in os.environ and "XP_HOST_THREADS" not in os.environ
    c = _lib.get_context(0)
    if not c.tables_loaded():
        c.tables_build()
    return c


@pytest.fixture
def make_ctx(monkeypatch):
    """A fresh context whose ``xp_create`` read ``XP_HOST_BLOCK_MB`` (and ``XP_HOST_THREADS``), tables built; closed
    at teardown."""
    made = []

    def make(block_mb=None, threads=None):
        for var, val in (("XP_HOST_BLOCK_MB", block_mb), ("XP_HOST_THREADS", threads)):
            if val is None:
                monkeypatch.delenv(var, raising=False)
            else:
                monkeypatch.setenv(var, str(val))
        c = _lib.Context(0)
        made.append(c)
        c.tables_build()
        return c

    yield make
    for c in made:
        c.close()


def host_form(a, form):
    """CPU tensor ``a`` ([L, N], or [N] for an explicit parcel) in one of the FORMS.  The slices are columns 3..3+N of
    a wider array whose other columns are NaN, so a copy with the wrong pitch or offset reads different values."""
    pin = form.startswith("pinned")
    if not form.endswith("slice"):
        out = torch.empty(a.shape, dtype=a.dtype, pin_memory=pin)
        out.copy_(a)
        return out
    n = a.shape[-1]
    wide = torch.full(tuple(a.shape[:-1]) + (n + 8,), float("nan"), dtype=a.dtype, pin_memory=pin)
    wide[..., 3:3 + n] = a
    return wide[..., 3:3 + n]


def axis_form(p, form, stride):
    """A shared 1-D pressure axis, pinned or not, with element stride ``stride``."""
    pin = form.startswith("pinned")
    wide = torch.full((p.shape[0] * stride,), float("nan"), dtype=p.dtype, pin_memory=pin)
    wide[::stride] = p
    return wide[::stride]


def pressure_with_own_stride(p, form):
    """Per-column pressure [L, N] as columns 5..5+N of an array 19 columns wider than N: its level stride differs
    from the temperature's in every form."""
    pin = form.startswith("pinned")
    L, n = p.shape
    wide = torch.full((L, n + 19), float("nan"), dtype=p.dtype, pin_memory=pin)
    wide[:, 5:5 + n] = p
    return wide[:, 5:5 + n]


def bits(x):
    return x.view({torch.float32: torch.int32, torch.float64: torch.int64, torch.int32: torch.int32}[x.dtype])


def assert_same_outputs(host, dev, what):
    for kind in dev:
        assert set(host[kind]) == set(dev[kind]), (what, kind)
        for f, d in dev[kind].items():
            h = host[kind][f]
            assert not h.is_cuda and h.dtype == d.dtype and h.shape == d.shape, (what, kind, f)
            hb, db = bits(h), bits(d.cpu())
            if not torch.equal(hb, db):
                bad = (hb != db).reshape(-1, hb.shape[-1]).any(0).nonzero().flatten()
                raise AssertionError(f"{what}: {kind}/{f} differs from the device path in {bad.numel()} columns, "
                                     f"first {bad[:6].tolist()}")


def host_vs_device(ctx, block_mb, p, t, td, kinds, what, options=None, profile=False, fields=None, shift=True,
                   explicit=None, pin_outputs=False, specific_humidity=False):
    """One call on the host arrays and the same call on CUDA copies, on ``ctx`` (created with ``block_mb`` MB blocks):
    outputs bit-identical, flags and ``last_exact_count`` equal, and the host call ran the blocks ``host_blocks``
    predicts, each with the launches of the device call.  Returns (flags, last_exact_count, blocks, launches per
    block)."""
    opts = options if options is not None else _lib.make_options()
    L, n = t.shape
    per_col = per_column_bytes(L, t.element_size(), p.dim() == 1, kinds, profile, fields, shift)
    expect_blocks = host_blocks(n, per_col, block_mb)[1]
    ex_d = None if explicit is None else tuple(e.cuda() for e in explicit)
    ctx.take_flags()
    out_d = ctx.alloc_outputs(t.cuda(), kinds, profile, fields=fields, shift=shift)
    n0 = ctx.launch_count()
    dev = ctx.cape_cin(p.cuda(), t.cuda(), td.cuda(), kinds=kinds, options=opts, explicit=ex_d, out=out_d,
                       specific_humidity=specific_humidity)
    dev_launches = ctx.launch_count() - n0
    dev_count = ctx.last_exact_count() if n else None
    dev_flags = ctx.take_flags()
    out_h = ctx.alloc_outputs(t, kinds, profile, pin_outputs=pin_outputs, fields=fields, shift=shift)
    for _, scal, sh, prof, _ in out_h.values():
        for x in (scal, prof):
            if x is not None:
                x.fill_(SENTINEL)
        if sh is not None:
            sh.fill_(-7)
        assert pin_outputs == scal.is_pinned()
    n0 = ctx.launch_count()
    host = ctx.cape_cin(p, t, td, kinds=kinds, options=opts, explicit=explicit, out=out_h,
                        specific_humidity=specific_humidity)
    host_launches = ctx.launch_count() - n0
    host_count = ctx.last_exact_count() if n else None
    host_flags = ctx.take_flags()
    assert_same_outputs(host, dev, what)
    assert host_flags == dev_flags, (what, host_flags, dev_flags)
    assert host_count == dev_count, (what, host_count, dev_count)
    # every block runs the launches of the one-block device call of the same route (2 to 4 kernels on the fast paths,
    # one exact kernel otherwise)
    if n == 0:
        assert host_launches == dev_launches == 0, what
        blocks = 0
    else:
        assert dev_launches >= 1 and host_launches % dev_launches == 0, (what, host_launches, dev_launches)
        blocks = host_launches // dev_launches
    assert blocks == expect_blocks, (what, blocks, expect_blocks)
    return host_flags, host_count, blocks, dev_launches


# --------------------------------------------------------------------------- the cases
@dataclass(frozen=True)
class Case:
    cols: str                   # key of COLUMNS
    dtype: torch.dtype
    pressure: str               # "pcol" | "pcol_stride" | "axis" | "axis_s2"
    kinds: tuple
    outputs: str                # key of OUTPUTS
    options: str                # key of OPTIONS
    in_form: str                # one of FORMS
    pin_outputs: bool
    blocks: int = 8             # target block count with 1 MB blocks; 0: the geometry in ``n`` / ``block_mb``
    n: int = 0
    block_mb: int = 1
    threads: int = None         # XP_HOST_THREADS (None: the library's default)
    sh: bool = False            # specific humidity in place of the dewpoint
    flag: str = None            # "dup": duplicate MU pressure, "top": NaN top temperature, in the last block


# regime columns: (source, regime, layout keywords)
COLUMNS = {
    "terrain": ("rc", "terrain", {}),
    "cold": ("rc", "cold", {}),
    "moist_heat": ("rc", "moist_heat", {}),
    "high_surface": ("rc", "high_surface", {}),
    "above_1100": ("rc", "above_1100", {}),
    "top0.01_L137": ("rc", "synth_like", dict(levels=137, p_top=0.01)),
    "era5": ("rc", "high_surface", dict(layout="era5")),
    "era5_masked": ("rc", "masked", dict(layout="era5_masked")),
    "axis": ("rc", "synth_like", dict(layout="axis", levels=50, p_top=5.0)),
    "synth_nan": ("synth", None, dict(levels=50, nan_columns=0.05, nan_levels=0.3, allnan_columns=0.02)),
}
OUTPUTS = {
    "all": dict(profile=False, fields=None, shift=True),
    "profile": dict(profile=True, fields=None, shift=True),
    "subset": dict(profile=False, fields=["cape", "cin", "lfc_pressure", "parcel_temperature"], shift=True),
    # no pointer that run_host checks for pageability: the outputs are copied straight to the caller's memory
    "absent": dict(profile=False, fields=["lcl_temperature", "el_temperature"], shift=False),
}
OPTIONS = {
    "default": dict(),
    "compat162": dict(metpy_compat="1.6.2"),
    "novtc": dict(virtual_temperature_correction=False),
    "exact": dict(exact_only=True),
}

# Pairwise cover: every value of every axis appears in at least one case of eight 1 MB blocks (each slot is reused at
# least twice, and pageable outputs of the first blocks are copied out by ``retire``).
CASES = {
    "terrain-f32-pcol-suite-profile": Case("terrain", torch.float32, "pcol", KINDS3, "profile", "default",
                                           "pageable", False),
    "cold-f64-pstride-ml": Case("cold", torch.float64, "pcol_stride", ("ml",), "all", "compat162", "pinned", False,
                                threads=1),
    "moist-f32-pcol-mu-q": Case("moist_heat", torch.float32, "pcol", ("mu",), "subset", "novtc", "pageable_slice",
                                True, threads=64, sh=True),
    "high-f32-pstride-sbmu-dup": Case("high_surface", torch.float32, "pcol_stride", ("sb", "mu"), "all", "default",
                                      "pinned_slice", False, flag="dup"),
    "above1100-f64-pcol-sbml-exact": Case("above_1100", torch.float64, "pcol", ("sb", "ml"), "profile", "exact",
                                          "pageable", True),
    "top0.01-f32-pcol-explicit": Case("top0.01_L137", torch.float32, "pcol", ("explicit",), "profile", "default",
                                      "pinned", False),
    "era5-f32-axis-suite-q": Case("era5", torch.float32, "axis", KINDS3, "all", "default", "pageable_slice", True,
                                  sh=True),
    "era5masked-f64-axis2-suite": Case("era5_masked", torch.float64, "axis_s2", KINDS3, "all", "default",
                                       "pinned_slice", True),
    "axis-f32-axis2-mlmu-absent": Case("axis", torch.float32, "axis_s2", ("ml", "mu"), "absent", "novtc", "pinned",
                                       False),
    "synth-f32-pcol-sb": Case("synth_nan", torch.float32, "pcol", ("sb",), "all", "compat162", "pinned_slice", False,
                              threads=1),
    "era5-f64-pcol-explicit-top": Case("era5", torch.float64, "pcol", ("explicit",), "subset", "novtc",
                                       "pageable_slice", True, flag="top"),
    "axis-f64-axis-sb-absent-exact": Case("axis", torch.float64, "axis", ("sb",), "absent", "exact", "pageable",
                                          False, threads=64),
    "terrain-f32-pcol-sbml-q": Case("terrain", torch.float32, "pcol", ("sb", "ml"), "all", "default", "pageable",
                                    False, sh=True),
    # one block at the default block size; fewer columns than a block; one column; none
    "era5-f32-axis-suite-1block": Case("era5", torch.float32, "axis", KINDS3, "all", "default", "pageable", False,
                                       blocks=0, n=5000, block_mb=DEFAULT_BLOCK_MB),
    "terrain-f32-pcol-sb-n700": Case("terrain", torch.float32, "pcol", ("sb",), "profile", "default", "pinned",
                                     False, blocks=0, n=700),
    "cold-f32-pcol-mu-n1": Case("cold", torch.float32, "pcol", ("mu",), "all", "default", "pageable_slice", True,
                                blocks=0, n=1),
    "synth-f64-pcol-explicit-n1": Case("synth_nan", torch.float64, "pcol", ("explicit",), "all", "exact",
                                       "pageable", False, blocks=0, n=1),
    "era5-f32-axis-suite-n0": Case("era5", torch.float32, "axis", KINDS3, "all", "default", "pageable", False,
                                   blocks=0, n=0),
}


def make_columns(name, n, seed):
    """float32 CPU tensors (p [L, N] or [L], T, Td [L, N]) of a COLUMNS entry."""
    src, regime, kw = COLUMNS[name]
    if src == "synth":
        kw = dict(kw)
        return synth.model_level_columns(n, kw.pop("levels"), seed=seed, **kw)
    p, t, td, _ = rc.columns(regime, n, seed, **kw)
    return torch.from_numpy(np.ascontiguousarray(p)), torch.from_numpy(t), torch.from_numpy(td)


def case_inputs(case, n, seed):
    """(p, T, Td, explicit) host tensors of ``case`` in its memory forms; flag columns in the last block."""
    p, t, td = make_columns(case.cols, n, seed)
    L = t.shape[0]
    if case.pressure.startswith("pcol") and p.dim() == 1:
        p = p[:, None].expand(L, n).contiguous()
    assert (p.dim() == 1) == case.pressure.startswith("axis"), case
    explicit = None
    if case.kinds == ("explicit",):
        k = 2                                                                   # the third level, warmed by 0.5 K
        pk = p[k].expand(n) if p.dim() == 1 else p[k]
        explicit = [pk.clone(), t[k] + 0.5, td[k].clone()]
    if case.sh:
        td = torch.from_numpy(rc.specific_humidity(p.numpy(), td.numpy()))
    if case.flag == "dup":
        # the most unstable parcel of column n-3 sits on a pressure that occurs twice (PF:130-131)
        c = n - 3
        p[1, c] = p[0, c]
        t[:2, c] = t[0, c] + 10.0
        td[:2, c] = t[0, c]
    if case.flag == "top":
        # column n-2 has data only on its top level (1 hPa, above the adiabat table): no level has both a parcel and
        # an environment temperature (PF:1149)
        t[:-1, n - 2] = float("nan")
        td[:-1, n - 2] = float("nan")
    t, td = t.to(case.dtype), td.to(case.dtype)
    p = p.to(case.dtype)
    if explicit is not None:
        explicit = [host_form(e.to(case.dtype), case.in_form) for e in explicit]
    t, td = host_form(t, case.in_form), host_form(td, case.in_form)
    if case.pressure == "pcol":
        p = host_form(p, case.in_form)
    elif case.pressure == "pcol_stride":
        p = pressure_with_own_stride(p, case.in_form)
        assert p.stride(0) != t.stride(0)
    else:
        p = axis_form(p, case.in_form, 2 if case.pressure == "axis_s2" else 1)
    return p, t, td, explicit


def case_size(case):
    """Columns of ``case``: ``blocks`` blocks of 1 MB, the last one partial (not a multiple of 1024 columns)."""
    if not case.blocks:
        return case.n
    _, _, kw = COLUMNS[case.cols]
    L = kw.get("levels", 37 if kw.get("layout", "").startswith("era5") else 70)
    es = 4 if case.dtype == torch.float32 else 8
    per_col = per_column_bytes(L, es, case.pressure.startswith("axis"), case.kinds, **OUTPUTS[case.outputs])
    c, _ = host_blocks(1 << 30, per_col, case.block_mb)
    return (case.blocks - 1) * c + c // 2 + 1


@pytest.mark.parametrize("name", list(CASES))
def test_host_path_equals_device_path(make_ctx, name):
    case = CASES[name]
    n = case_size(case)
    ctx = make_ctx(case.block_mb, case.threads)
    p, t, td, explicit = case_inputs(case, n, seed=7000 + list(CASES).index(name))
    if case.in_form.startswith("pinned"):
        assert t.is_pinned() and td.is_pinned() and p.is_pinned()
    if case.in_form.endswith("slice") and n > 1:
        assert t.stride(0) > n
    flags, _, ran, _ = host_vs_device(ctx, case.block_mb, p, t, td, case.kinds, name,
                                      options=_lib.make_options(**OPTIONS[case.options]), explicit=explicit,
                                      pin_outputs=case.pin_outputs, specific_humidity=case.sh, **OUTPUTS[case.outputs])
    assert ran == (case.blocks or (1 if n else 0)), ran
    if case.flag == "dup":
        assert flags & _lib.FLAG_PRESSURES_NOT_UNIQUE, flags
    if case.flag == "top":
        assert flags & _lib.FLAG_TOP_TEMPERATURE_NAN, flags


def test_cases_cover_every_value_with_many_blocks():
    """Every value of every axis appears in a case of at least seven blocks (CPU-side check of the case list)."""
    many = [c for c in CASES.values() if c.blocks >= 7]
    axes = {"cols": COLUMNS, "dtype": (torch.float32, torch.float64), "pressure": ("pcol", "pcol_stride", "axis",
                                                                                    "axis_s2"),
            "outputs": OUTPUTS, "options": OPTIONS, "in_form": FORMS, "pin_outputs": (False, True),
            "threads": (None, 1, 64), "sh": (False, True), "flag": (None, "dup", "top")}
    for axis, values in axes.items():
        for v in values:
            assert any(getattr(c, axis) == v for c in many), (axis, v)
    kinds = {c.kinds for c in many}
    for k in [("sb",), ("ml",), ("mu",), ("sb", "ml"), ("sb", "mu"), ("ml", "mu"), KINDS3, ("explicit",)]:
        assert k in kinds, k


# --------------------------------------------------------------------------- one context, changing calls
def test_one_context_through_growing_and_shrinking_calls(make_ctx):
    """Slot and mirror buffers are re-allocated as the bytes per column grow and shrink and the pinned / pageable mix
    changes; every call still equals its device call."""
    ctx = make_ctx(1)

    def era5(n, seed, dtype=torch.float32, form="pageable"):
        p, t, td = synth.era5_columns(n, seed=seed)
        return axis_form(p.to(dtype), form, 1), host_form(t.to(dtype), form), host_form(td.to(dtype), form)

    def model(n, seed, form):
        p, t, td = synth.model_level_columns(n, 70, seed=seed)
        return [host_form(x, form) for x in (p, t, td)]

    # 1. small pinned call, 2. large pageable call with profiles, 3. small pageable call, 4. float64, 5. large pinned
    steps = [("small pinned", era5(3000, 1, form="pinned"), KINDS3, dict(pin_outputs=True), 2),
             ("large pageable profiles", model(9000, 2, "pageable"), KINDS3, dict(profile=True), 9),
             ("small pageable", era5(2500, 3), ("sb",), {}, 2),
             ("float64", era5(20000, 4, torch.float64, "pageable_slice"), KINDS3, {}, 20),
             ("large pinned", model(30000, 5, "pinned"), ("sb", "mu"), dict(pin_outputs=True), 30)]
    for what, (p, t, td), kinds, kw, blocks in steps:
        _, _, ran, _ = host_vs_device(ctx, 1, p, t, td, kinds, what, **kw)
        assert ran == blocks, (what, ran)


# --------------------------------------------------------------------------- the fix-up count of a host call
@pytest.mark.parametrize("route", ["pcol_table", "pcol_gather", "axis", "exact_only", "f64_pcol"])
def test_last_exact_count_sums_every_block(make_ctx, route):
    """After a host call ``last_exact_count`` is the hand-over count of the whole call, not of its last block: equal to
    the device call on the same columns with 1 MB blocks; -1 where no block took the fast path."""
    ctx = make_ctx(1)
    layout = {"axis": dict(layout="era5")}.get(route, {})
    p, t, td, _ = rc.columns("high_surface", 20_000, seed=81, **layout)
    p, t, td = [torch.from_numpy(np.ascontiguousarray(x)) for x in (p, t, td)]
    if route == "f64_pcol":
        p, t, td = p.double(), t.double(), td.double()
    kinds = ("sb",) if route == "pcol_gather" else KINDS3
    opts = _lib.make_options(exact_only=route == "exact_only")
    _, count, blocks, launches = host_vs_device(ctx, 1, p, t, td, kinds, route, options=opts)
    assert blocks >= 7, blocks
    # launches per block: table route 3, gather route 2, shared axis 4, the exact kernel 1
    assert launches == {"pcol_table": 3, "pcol_gather": 2, "axis": 4}.get(route, 1), launches
    if route in ("exact_only", "f64_pcol"):
        assert count == -1
    else:
        assert count > 0, count


# --------------------------------------------------------------------------- the public surface at its default blocks
def test_parcel_suite_on_pageable_numpy_at_default_blocks(global_context):
    """``parcel_suite`` on pageable NumPy ERA5 arrays -- what a user of the reference's API gets -- over four default
    192 MB blocks (the outputs of the first block are copied out when its slot is reused), bit for bit against
    ``parcel_suite`` on CUDA tensors of the same arrays."""
    import xarray_parcel_b200.parcel_functions as pf
    n = 1_400_000
    per_col = per_column_bytes(37, 4, True, KINDS3)
    assert per_col == 452
    c, blocks = host_blocks(n, per_col, DEFAULT_BLOCK_MB)
    assert (c, blocks) == (444_416, 4)
    p, t, td = synth.era5_columns(n, seed=90, device="cuda")
    P, T, D = p.cpu().numpy(), t.cpu().numpy(), td.cpu().numpy()
    ctx = global_context
    n0 = ctx.launch_count()
    dev = pf.parcel_suite(p, t, td)
    dev_launches = ctx.launch_count() - n0
    n0 = ctx.launch_count()
    host = pf.parcel_suite(P, T, D)
    assert ctx.launch_count() - n0 == blocks * dev_launches
    assert set(host) == set(dev)
    for k in dev:
        a = np.asarray(host[k])
        assert isinstance(a, np.ndarray) and a.dtype == np.float32, k
        assert np.array_equal(a.view(np.int32), dev[k].cpu().numpy().view(np.int32)), k


# --------------------------------------------------------------------------- streaming against one device call
@pytest.mark.parametrize("workers", [1, 3])
def test_streamed_blocks_equal_one_device_call(tmp_path, monkeypatch, global_context, workers):
    """``parcel_suite_chunks`` / ``streaming.suite_blocks`` over strided views of memory-mapped files, on contexts with
    1 MB blocks, against ONE device-tensor call over the whole array (not against the host path itself)."""
    import xarray_parcel_b200.parcel_functions as pf
    from xarray_parcel_b200 import streaming
    monkeypatch.setenv("XP_HOST_BLOCK_MB", "1")         # read when suite_blocks creates its contexts
    if workers == 1:
        # ERA5 levels, specific humidity, parcel_suite_chunks
        p, t, td, _ = rc.columns("moist_heat", 60_000, seed=91, layout="era5")
        q = rc.specific_humidity(p, td)
        arrays, kinds, fields, sh = (t, q), KINDS3, None, True
    else:
        # per-column pressure on model levels, a subset of the fields, streaming.suite_blocks
        p, t, td, _ = rc.columns("terrain", 30_000, seed=92)
        arrays, kinds, fields, sh = (p, t, td), ("sb", "mu"), ["cape", "cin", "el_pressure"], False
    maps = []
    for i, a in enumerate(arrays):
        path = os.path.join(tmp_path, f"a{i}.npy")
        np.save(path, a)
        maps.append(np.load(path, mmap_mode="c"))          # writable views: handed to the library without a copy
    if workers == 1:
        P, T, D = p, maps[0], maps[1]
    else:
        P, T, D = maps
    blocks = list(streaming.iter_column_blocks(P, T, D, 7_777))
    assert blocks[1][1].strides[0] == T.strides[0] and not blocks[1][1].flags.c_contiguous
    ctx = global_context
    dev_in = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (p, *arrays[-2:])]
    opts = _lib.make_options()
    dev = ctx.cape_cin(*dev_in, kinds=kinds, options=opts, specific_humidity=sh)
    if workers == 1:
        parts = list(pf.parcel_suite_chunks(blocks, workers=workers, specific_humidity=True))
        names = {"sb": "surface", "ml": "mixed_100", "mu": "max"}
        for kind in kinds:
            parcel = ["parcel_pressure", "parcel_temperature", "parcel_dewpoint"] if kind != "sb" else []
            for f in ["cape", "cin"] + pf._SCALAR_VARS + parcel:
                got = np.concatenate([d[f"{names[kind]}_{f}"] for d in parts])
                assert np.array_equal(got.view(np.int32), dev[kind][f].cpu().numpy().view(np.int32)), (kind, f)
    else:
        parts = list(streaming.suite_blocks(blocks, kinds=kinds, workers=workers, options=opts, fields=fields))
        for kind in kinds:
            assert set(parts[0][kind]) == set(fields) | {"level_shift"}
            for f in fields + ["level_shift"]:
                got = torch.cat([d[kind][f] for d in parts])
                assert torch.equal(bits(got), bits(dev[kind][f].cpu())), (kind, f)


# --------------------------------------------------------------------------- explicit parcels against the oracle
@pytest.mark.parametrize("regime", ["terrain", "era5_masked"])
def test_explicit_parcel_host_path_matches_oracle(make_ctx, regime):
    """Explicit parcels (a level of each column, warmed by 0.5 K) through the host path in 1 MB blocks: float64
    against the oracle at 1e-9 (the knife-edge allowance of test_gpu_parity._check), float32 equal to the device path
    (which test_gpu_regimes pins to its own float64 results)."""
    ctx = make_ctx(1)
    kw = dict(layout="era5_masked") if regime == "era5_masked" else {}
    p, t, td, _ = rc.columns("masked" if regime == "era5_masked" else regime, 3000, seed=95, **kw)
    P, T, D = [torch.from_numpy(np.ascontiguousarray(x)) for x in (p, t, td)]
    k = 4
    pp = P[k].expand(T.shape[1]).clone() if P.dim() == 1 else P[k].clone()
    ex = [pp, T[k] + 0.5, D[k].clone()]
    # float32: the host path equals the device path
    host_vs_device(ctx, 1, P, T, D, ("explicit",), f"{regime} f32", explicit=ex, profile=True)
    # float64: the host path against the oracle
    P64, T64, D64 = P.double(), T.double(), D.double()
    ex64 = [e.double() for e in ex]
    per_col = per_column_bytes(T.shape[0], 8, P.dim() == 1, ("explicit",))
    assert host_blocks(T.shape[1], per_col, 1)[1] >= 2
    res = ctx.cape_cin(P64, T64, D64, kinds=("explicit",), explicit=ex64)["explicit"]
    ctx.take_flags()
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    opts = op.Options(op.MoistLapseLUT(otab.AdiabatTables(pl, tl, idx, cur)), lcl_mode="converged")
    Pn = P64.numpy() if P64.dim() == 2 else np.broadcast_to(P64.numpy()[:, None], T64.shape)
    cc, prof = op.cape_cin(Pn, T64.numpy(), D64.numpy(), *(e.numpy() for e in (ex64[1], ex64[0], ex64[2])), opts)
    ora = {"x_" + key: v for key, v in {**cc, **prof}.items() if v.ndim == 1}
    _check(res, ora, "x_", 1e-9, what=f"{regime} explicit host path: ", knife=(ex64[1] == ex64[2]).numpy())
