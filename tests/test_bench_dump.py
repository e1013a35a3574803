"""bench.py --dump-outputs: every output of the timed step as <kind>_<field>.npy, undefined (NaN) entries as 0 beside a
<kind>_<field>_defined.npy mask; a set larger than the size cap is cut to one seeded sample of columns, the same in every
file and from call to call."""

import os

import numpy as np
import torch

import bench


def _column_numbered_outputs(n, L, profile):
    """Output blocks laid out like Context.alloc_outputs whose every value is its column number, except in columns
    divisible by 7, where the value is undefined (NaN) as an absent LFC / EL is."""
    col = torch.arange(n, dtype=torch.float32)
    col[::7] = float("nan")
    outs = {}
    for kind in ("sb", "mu"):
        names = bench.BENCH_FIELDS[kind]
        scal = col.expand(len(names), n).contiguous()
        prof = col.expand(6, L + 1, n).contiguous() if profile else None
        outs[kind] = (None, scal, None, prof, names)
    return outs


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _check_finite_with_masks(got, cols):
    """Every file is finite; each output equals its column numbers where defined, 0 elsewhere, and its mask says which."""
    values = {k: v for k, v in got.items() if not k.endswith("_defined")}
    assert set(got) == set(values) | {k + "_defined" for k in values}
    defined = cols % 7 != 0
    for name, a in values.items():
        m = got[name + "_defined"]
        assert a.dtype == np.float32 and m.dtype == np.float32
        assert np.isfinite(a).all() and np.isfinite(m).all(), name
        assert np.array_equal(m, np.broadcast_to(defined.astype(np.float32), m.shape)), name
        assert np.array_equal(a, np.broadcast_to(np.where(defined, cols, 0).astype(np.float32), a.shape)), name
    return values


def test_small_output_sets_are_written_whole(tmp_path):
    n, L = 1000, 5
    bench.dump_outputs(str(tmp_path), _column_numbered_outputs(n, L, profile=True), n)
    values = _check_finite_with_masks(_load(tmp_path), np.arange(n))
    assert len(values) == len(bench.BENCH_FIELDS["sb"]) + len(bench.BENCH_FIELDS["mu"]) + 2 * 6
    assert set(values) >= {"sb_cape", "mu_parcel_dewpoint", "mu_profile_pressure"}
    for name, a in values.items():
        assert a.shape == ((L + 1, n) if "profile" in name else (n,))


def test_large_output_sets_are_one_seeded_column_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    n, L = 20_000, 3
    per_column = 2 * (len(bench.BENCH_FIELDS["sb"]) + len(bench.BENCH_FIELDS["mu"]) + 2 * 6 * (L + 1)) * 4
    dumps = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _column_numbered_outputs(n, L, profile=True), n)
        dumps.append(_load(tmp_path / d))
    # the sample's column numbers, recovered from a value file and its mask (undefined columns are multiples of 7)
    a, m = dumps[0]["sb_cape"], dumps[0]["sb_cape_defined"]
    cols = np.where(m == 1, a, np.nan)
    assert cols.size == bench.DUMP_BYTES // per_column
    known = cols[~np.isnan(cols)]
    assert np.all(np.diff(known) > 0) and known[0] >= 0 and known[-1] < n
    assert sum(x.nbytes for x in dumps[0].values()) <= bench.DUMP_BYTES
    for name, x in dumps[0].items():
        assert np.array_equal(x, np.broadcast_to(dumps[0]["sb_cape" + ("_defined" if name.endswith("_defined") else "")],
                                                 x.shape)), name
        assert np.array_equal(x, dumps[1][name]), name
    assert np.isfinite(np.concatenate([x.ravel() for x in dumps[0].values()])).all()
