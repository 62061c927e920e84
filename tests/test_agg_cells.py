"""Narrow cells of the flat GROUP BY kernel's shared-memory table: u32 COUNT(*) / non-null counters, Int64 MIN / MAX as
u32 offsets from a base the footer statistics give, f64 sums of the hot groups without per-lane cells sent to L2.
Every case is checked against the oracle, including files whose statistics are missing or understate the range."""
import os
import struct
import subprocess
import sys

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest

from oracle.oracle import Oracle
from parseable_b200.query import StandardTableProvider, count, count_star, max_, min_, sum_

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64_REL = 1e-9

AGGS = [count_star(), min_("v"), max_("v"), sum_("v"), sum_("f"), count("v"), max_("f"), min_("t")]


def _table(n, groups, v, null_rate=0.0, seed=7):
    """Zipf-skewed string keys (the hottest take per-lane cells, the next ones hot cells, the tail cold ones)."""
    rng = np.random.default_rng(seed)
    g = np.minimum(rng.zipf(1.1, n) - 1, groups - 1)
    mask = (rng.random(n) < null_rate) if null_rate else None
    return pa.table({
        "g": pa.array([f"k{x:06d}" for x in g]).dictionary_encode(),
        "v": pa.array(v, type=pa.int64(), mask=mask),
        "f": pa.array(rng.random(n) * 100.0, mask=mask),
        "t": pa.array(rng.integers(-50, 50, n), type=pa.int64()),
    })


def _write(t, path, **kw):
    pq.write_table(t, path, compression="NONE", row_group_size=100_000, data_page_size=1 << 20, **kw)
    return path


def _patch_footer_i64(path, old: int, new: int) -> int:
    """Rewrite an Int64 statistics value inside the footer only (the pages keep the real values): statistics that lie."""
    data = bytearray(open(path, "rb").read())
    flen = struct.unpack("<I", data[-8:-4])[0]
    start = len(data) - 8 - flen
    footer = bytes(data[start:-8])
    n = footer.count(struct.pack("<q", old))
    data[start:-8] = footer.replace(struct.pack("<q", old), struct.pack("<q", new))
    open(path, "wb").write(bytes(data))
    return n


def _check(path, aggs=AGGS):
    ora = Oracle.from_parquet(path)
    prov = StandardTableProvider([path], schema=ora.table.schema)
    got = prov.aggregate(["g"], aggs).table().sort_by("g")
    exp = ora.group_by(["g"], aggs).sort_by("g")
    assert got.num_rows == exp.num_rows
    for name in exp.column_names:
        a, b = got[name].to_pylist(), exp[name].to_pylist()
        if name.startswith("sum(f"):
            assert all((x is None) == (y is None) and (x is None or abs(x - y) <= F64_REL * abs(y)) for x, y in zip(a, b)), name
        else:
            assert a == b, name
    return got


def test_narrow_range_many_groups(data_dir, built):
    """values inside a 2^16 window, 20 000 possible groups: per-lane, hot and cold cells in one query"""
    n = 400_000
    rng = np.random.default_rng(1)
    p = _write(_table(n, 20_000, rng.integers(1_000_000, 1_065_536, n)), os.path.join(data_dir, "cells_many.parquet"))
    got = _check(p)
    assert got.num_rows > 3000


def test_negative_values(data_dir, built):
    n = 300_000
    rng = np.random.default_rng(2)
    p = _write(_table(n, 500, rng.integers(-(2**31) - 5, -(2**31) + 70_000, n)), os.path.join(data_dir, "cells_neg.parquet"))
    _check(p)


def test_range_wider_than_u32_keeps_8_byte_cells(data_dir, built):
    n = 300_000
    rng = np.random.default_rng(3)
    v = rng.integers(-(2**40), 2**40, n)
    v[:3] = [-(2**63), 2**63 - 1, 0]
    p = _write(_table(n, 2_000, v), os.path.join(data_dir, "cells_wide.parquet"))
    _check(p)


def test_window_at_the_top_of_int64(data_dir, built):
    """a narrow range ending at INT64_MAX: the window must not wrap"""
    n = 200_000
    rng = np.random.default_rng(4)
    p = _write(_table(n, 1_000, (2**63 - 1) - rng.integers(0, 1000, n)), os.path.join(data_dir, "cells_top.parquet"))
    _check(p)


def test_missing_statistics(data_dir, built):
    n = 200_000
    rng = np.random.default_rng(5)
    p = _write(_table(n, 1_000, rng.integers(0, 5_000, n)), os.path.join(data_dir, "cells_nostats.parquet"), write_statistics=False)
    assert pq.ParquetFile(p).metadata.row_group(0).column(1).statistics is None
    _check(p)


def test_statistics_that_understate_the_range(data_dir, built):
    """the footer claims [0, 4999]; a few rows in several groups lie far outside on both sides: they must still win"""
    n = 300_000
    rng = np.random.default_rng(6)
    v = rng.integers(0, 5_000, n)
    lo, hi = -7_000_000_000_321, 9_000_000_000_123
    v[rng.choice(n, 40, replace=False)] = lo
    v[rng.choice(n, 40, replace=False)] = hi
    v[:2] = [0, 4_999]
    p = _write(_table(n, 300, v), os.path.join(data_dir, "cells_lying.parquet"))
    assert _patch_footer_i64(p, hi, 4_999) > 0 and _patch_footer_i64(p, lo, 0) > 0
    md = pq.ParquetFile(p).metadata
    for r in range(md.num_row_groups):
        st = md.row_group(r).column(1).statistics
        assert st.min >= 0 and st.max <= 4_999
    got = _check(p)
    assert min(got["min(v)"].to_pylist()) == lo and max(got["max(v)"].to_pylist()) == hi


def test_null_inputs(data_dir, built):
    """NULL inputs: the u32 non-null counters, and groups whose values are all NULL"""
    n = 300_000
    rng = np.random.default_rng(8)
    p = _write(_table(n, 3_000, rng.integers(100, 900, n), null_rate=0.3), os.path.join(data_dir, "cells_nulls.parquet"))
    _check(p)


def test_two_rank_allreduce_with_understated_statistics(small_files, tmp_path, built):
    """two ranks, each with its own narrow window; rank 1's footers understate latency_ms"""
    from parseable_b200 import _lib as L
    if L.load().pq_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from parseable_b200 import synth
    split = []
    for tag, rate, rg in (("nn", 0.0, 3), ("nulls", 0.02, 9)):
        p = str(tmp_path / f"cells_{tag}.parquet")
        synth.write_logs16(p, n_row_groups=1, first_rg=rg, rows_per_group=50_000, null_rate=rate)
        split.append(p)
    col = pq.ParquetFile(split[1]).schema_arrow.get_field_index("latency_ms")
    true_max = pq.ParquetFile(split[1]).metadata.row_group(0).column(col).statistics.max
    assert _patch_footer_i64(split[1], true_max, 10) > 0
    assert pq.ParquetFile(split[1]).metadata.row_group(0).column(col).statistics.max == 10
    idfile = str(tmp_path / "nccl_id")
    procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "scripts", "mgpu_check.py"), str(r), "2", idfile,
                               small_files["nn"], "--"] + split, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r}:\n{o[-3000:]}"
        assert "parity OK" in o
