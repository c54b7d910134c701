"""Session ops on the B200 against the CPU oracle (oracle/sessions.py): Groupby over every key
type and aggregation, ListSlice over ragged lists with null leaves, a 10^8-row partition, and the
Categorify -> Groupby -> ListSlice pipeline of the Transformers4Rec example (reference
tests/unit/test_tf4rec.py:141-200) on a key-shuffled, partitioned Dataset."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pandas as pd
import pytest

from oracle import sessions as osess

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL_AGGS = ["count", "sum", "mean", "min", "max", "std", "var", "median", "nunique", "list", "first", "last"]
FLOAT_RTOL = {"sum": 1e-6, "mean": 1e-6, "median": 1e-6, "std": 1e-5, "var": 1e-5}


@pytest.fixture(scope="module")
def nvt():
    import nvtabular
    return nvtabular


def _keys(rng, kind, n, n_groups):
    g = rng.integers(0, n_groups, n)
    null = rng.random(n) < 0.05
    if kind == "int32":
        return {"k": pd.array(np.where(null, None, g - n_groups // 2), dtype="Int32")}
    if kind == "int64":
        return {"k": pd.array(np.where(null, None, (g - n_groups // 2) * (1 << 40)), dtype="Int64")}
    if kind == "float64":
        return {"k": np.where(null, np.nan, (g - n_groups // 2) * 0.25)}
    if kind == "string":
        return {"k": pd.Series([None if m else f"s{v:05d}" for v, m in zip(g, null)], dtype=object)}
    if kind == "bool":                   # plain bool: the other key types carry the null keys
        return {"k": g % 2 == 0}
    return {"k": pd.array(np.where(null, None, g % 7), dtype="Int32"),       # two-column keys
            "k2": pd.Series([None if m else f"t{v % 13}" for v, m in zip(g, rng.random(n) < 0.03)], dtype=object)}


def _frame(rng, kind, n, n_groups):
    df = pd.DataFrame(_keys(rng, kind, n, n_groups))
    df["ts"] = pd.array(np.where(rng.random(n) < 0.05, None, rng.integers(0, 50, n)), dtype="Int64")
    df["x"] = np.where(rng.random(n) < 0.1, np.nan, rng.normal(3.0, 2.0, n))
    df["i"] = pd.array(np.where(rng.random(n) < 0.1, None, rng.integers(-1000, 1000, n)), dtype="Int32")
    return df


def _f(v):
    return pd.to_numeric(pd.Series(list(v), dtype=object), errors="coerce").to_numpy(dtype=float)


def _assert_column(got, exp, name, agg):
    assert len(got) == len(exp), name
    if agg == "list" or (len(exp) and isinstance(exp.iloc[0], (list, np.ndarray))):
        for a, b in zip(got, exp):
            np.testing.assert_array_equal(_f(a), _f(b), err_msg=name)
        return
    is_str = any(isinstance(v, str) for v in exp)
    g = got.to_numpy(dtype=object) if is_str else _f(got)
    e = exp.to_numpy(dtype=object) if is_str else _f(exp)
    if agg in FLOAT_RTOL:
        np.testing.assert_allclose(g, e, rtol=FLOAT_RTOL[agg], atol=1e-6, equal_nan=True, err_msg=name)
    elif g.dtype == object:
        assert list(pd.Series(g).where(pd.notna(g), None)) == list(pd.Series(e).where(pd.notna(e), None)), name
    else:
        np.testing.assert_array_equal(g, e, err_msg=name)


def _compare(got: pd.DataFrame, exp: pd.DataFrame, sep="-"):
    assert list(got.columns) == list(exp.columns)
    for c in exp.columns:
        agg = c.rsplit(sep, 1)[1] if sep in c else None
        _assert_column(got[c].reset_index(drop=True), exp[c].reset_index(drop=True), c, agg)


@pytest.mark.parametrize("kind", ["int32", "int64", "float64", "string", "bool", "two"])
@pytest.mark.parametrize("ascending", [True, False])
def test_groupby_random_against_oracle(nvt, kind, ascending):
    rng = np.random.default_rng(zlib.crc32(f"{kind}{ascending}".encode()))
    n_groups = 3 if kind == "bool" else 400
    df = _frame(rng, kind, 6000, n_groups)
    keys = ["k", "k2"] if kind == "two" else ["k"]
    aggs = {"x": ALL_AGGS, "i": ALL_AGGS, "ts": ["first", "last", "list", "min", "max"]}
    if kind == "two":
        aggs["k"] = ["count"]                     # a key column is never aggregated (_get_agg_dicts)
    op = nvt.ops.Groupby(groupby_cols=keys, sort_cols=["ts"], aggs=aggs, name_sep="-", ascending=ascending)
    wf = nvt.Workflow(list(df.columns) >> op)
    got = wf.fit_transform(nvt.Dataset(df)).to_ddf().compute()
    exp = osess.groupby(df, keys, ["ts"], aggs, name_sep="-", ascending=ascending)
    _compare(got, exp)
    assert wf.output_schema["x-list"].is_list and wf.output_schema["x-list"].is_ragged
    assert str(got["x-count"].dtype) == "int32" and str(got["x-mean"].dtype) == "float32"


def test_groupby_without_sort_cols_keeps_input_order(nvt):
    rng = np.random.default_rng(5)
    df = pd.DataFrame({"k": rng.integers(0, 30, 3000), "v": rng.integers(0, 10**6, 3000)})
    for ascending in (True, False):
        op = nvt.ops.Groupby(groupby_cols="k", aggs=["list", "first", "last"], ascending=ascending)
        got = nvt.Workflow(["k", "v"] >> op).fit_transform(nvt.Dataset(df)).to_ddf().compute()
        _compare(got, osess.groupby(df, ["k"], None, ["list", "first", "last"], ascending=ascending), sep="_")


def test_groupby_single_rows_empty_partition_and_one_huge_group(nvt):
    rng = np.random.default_rng(11)
    n = 1 << 24
    k = rng.integers(1, n // 4, n)                 # mostly single-row and short groups
    k[rng.random(n) < 0.12] = 0                    # one group with > 10 % of the rows
    df = pd.DataFrame({"k": k, "ts": rng.integers(0, 1 << 30, n),
                       "x": np.where(rng.random(n) < 0.05, np.nan, rng.normal(0, 1, n)).astype(np.float32)})
    aggs = {"x": [a for a in ALL_AGGS if a != "list"], "ts": ["first", "last", "count"]}
    op = nvt.ops.Groupby(groupby_cols="k", sort_cols="ts", aggs=aggs, name_sep="-")
    got = nvt.Workflow(["k", "ts", "x"] >> op).fit_transform(nvt.Dataset(df)).to_ddf().compute()
    # pandas' grouped var / std of a float32 column accumulate in float32 (1e-3 off on this group);
    # the float64 copy holds the same values
    exp = osess.groupby(df.astype({"x": "float64"}), ["k"], ["ts"], aggs, name_sep="-")
    assert got["x-count"].iloc[0] > n // 10
    _compare(got, exp)

    empty = df.iloc[:0]
    wf = nvt.Workflow(["k", "ts", "x"] >> nvt.ops.Groupby(groupby_cols="k", sort_cols="ts", aggs=aggs, name_sep="-"))
    out = wf.fit_transform(nvt.Dataset(empty)).to_ddf().compute()
    assert len(out) == 0 and list(out.columns) == list(exp.columns)
    assert str(out["x-count"].dtype) == "int32" and str(out["x-min"].dtype) == "float32"


def test_groupby_list_first_last(nvt):
    """reference tests/unit/ops/test_groupyby.py::test_groupby_list_first_last"""
    df = pd.DataFrame({"user_id": [1, 1, 2, 3], "user_vector": [[1, 2, 3], [4, 5, 6], [2, 2, 3], [3, 2, 3]]})
    out = nvt.Workflow(list(df.columns) >> nvt.ops.Groupby(groupby_cols="user_id",
                                                            aggs={"user_vector": ["first", "last"]})
                       ).fit_transform(nvt.Dataset(df)).compute()
    assert [list(r) for r in out["user_vector_first"]] == [[1, 2, 3], [2, 2, 3], [3, 2, 3]]
    assert [list(r) for r in out["user_vector_last"]] == [[4, 5, 6], [2, 2, 3], [3, 2, 3]]


def _ragged(rng, n, max_len=12):
    rows = []
    for _ in range(n):
        L = int(rng.integers(0, max_len))
        vals = rng.integers(-100, 100, L).astype(float)
        vals[rng.random(L) < 0.1] = np.nan
        rows.append(list(vals))
    return rows


@pytest.mark.parametrize("start,end", [(3, None), (-3, None), (0, None), (2, 7), (-5, -1), (-2, 4), (3, -2),
                                       (-7, -8), (20, 30)])
@pytest.mark.parametrize("pad", [False, True])
def test_list_slice_random_against_oracle(nvt, start, end, pad):
    from nvtabular_b200.column import Column, DeviceFrame
    rng = np.random.default_rng(abs(start * 31 + (end or 0)))
    rows = _ragged(rng, 3000)
    _, _, max_el = osess.list_slice_bounds(start, end)
    if pad and not 0 <= max_el < osess.INT64_MAX:
        with pytest.raises(ValueError):
            nvt.ops.ListSlice(start, end, pad=True)
        return
    op = nvt.ops.ListSlice(start, end, pad=pad, pad_value=-7)
    frame = DeviceFrame({"y": Column.from_lists(rows)})
    got = op.transform(nvt.ColumnSelector(["y"]), frame)["y"].to_pandas()
    exp = osess.list_slice(rows, start, end, pad=pad, pad_value=-7)
    assert len(got) == len(exp)
    for a, b in zip(got, exp):
        np.testing.assert_array_equal(np.asarray(a, dtype=float), np.asarray(b, dtype=float))


def test_groupby_at_scale_1e8_rows(nvt):
    """10^8 rows, ~10^7 sessions: every group's count, and 10^4 sampled groups in full"""
    import torch
    from nvtabular_b200.column import Column, DeviceFrame
    rng = np.random.default_rng(2024)
    n, n_groups = 100_000_000, 10_000_000
    key = rng.integers(0, n_groups, n, dtype=np.int64) * 7919
    ts = rng.integers(0, 1 << 40, n, dtype=np.int64)
    price = rng.random(n, dtype=np.float32)
    frame = DeviceFrame({"s": Column(torch.from_numpy(key).cuda()), "ts": Column(torch.from_numpy(ts).cuda()),
                         "p": Column(torch.from_numpy(price).cuda())})
    op = nvt.ops.Groupby(groupby_cols="s", sort_cols="ts", aggs={"p": ["list", "count", "mean", "min", "max"],
                                                                 "ts": ["first", "last"]}, name_sep="-")
    out = op.transform(nvt.ColumnSelector(["s", "ts", "p"]), frame)
    uniq, counts = np.unique(key, return_counts=True)
    np.testing.assert_array_equal(out["s"].data.cpu().numpy(), uniq)
    np.testing.assert_array_equal(out["p-count"].data.cpu().numpy(), counts)
    del frame
    pick = np.sort(rng.choice(len(uniq), 10_000, replace=False))
    sel = np.isin(key, uniq[pick])
    exp = osess.groupby(pd.DataFrame({"s": key[sel], "ts": ts[sel], "p": price[sel]}), ["s"], ["ts"],
                        {"p": ["list", "count", "mean", "min", "max"], "ts": ["first", "last"]}, name_sep="-")
    off = out["p-list"].offsets.cpu().numpy()
    leaves = out["p-list"].data.cpu().numpy()
    got = {"s": uniq[pick], "p-list": [leaves[off[g]:off[g + 1]] for g in pick]}
    for c in ("p-count", "p-mean", "p-min", "p-max", "ts-first", "ts-last"):
        got[c] = out[c].data.cpu().numpy()[pick]
    _compare(pd.DataFrame({k: pd.Series(list(v), dtype=object) if k == "p-list" else v for k, v in got.items()}), exp)


def _sessions_frame(rng, n):
    return pd.DataFrame({
        "session_id": rng.integers(0, n // 8, n),
        "item_id": pd.Series([f"item{v}" for v in rng.zipf(1.3, n) % 5000], dtype=object),
        "ts": rng.integers(0, 10_000, n),
        "price": np.where(rng.random(n) < 0.05, np.nan, rng.gamma(2.0, 10.0, n)),
    })


def test_session_pipeline_on_shuffled_partitions(nvt, tmp_path):
    """Categorify -> Groupby -> ListSlice(pad=True), Normalize fitted on the grouped rows, on four
    partitions after shuffle_by_keys == the oracle on the whole frame"""
    from oracle.categorify import CategorifyOracle
    rng = np.random.default_rng(7)
    df = _sessions_frame(rng, 40_000)
    ops = nvt.ops
    cats = ["item_id"] >> ops.Categorify(out_path=str(tmp_path))
    aggs = {"item_id": ["list", "count"], "price": ["list", "mean"], "ts": ["first", "last"]}
    sessions = (["session_id", "ts", "price"] + cats) >> ops.Groupby(
        groupby_cols=["session_id"], sort_cols=["ts"], aggs=aggs, name_sep="-")
    seqs = sessions["item_id-list", "price-list"] >> ops.ListSlice(-20, pad=True)
    normed = sessions["price-mean"] >> ops.FillMissing(0.0) >> ops.Normalize()
    wf = nvt.Workflow(sessions["session_id", "item_id-count", "ts-first", "ts-last"] + seqs + normed)
    ds = nvt.Dataset(df, npartitions=4).shuffle_by_keys(["session_id"])
    assert ds.npartitions == 4
    got = wf.fit_transform(ds).to_ddf().compute().sort_values("session_id", ignore_index=True)

    enc = df.copy()
    enc["item_id"] = CategorifyOracle(["item_id"]).fit(df).transform(df)["item_id"].to_numpy()
    exp = osess.groupby(enc, ["session_id"], ["ts"], aggs, name_sep="-")
    for c in ("item_id-list", "price-list"):
        exp[c] = pd.Series(osess.list_slice(exp[c], -20, pad=True), dtype=object)
    pm = exp["price-mean"].astype("float32").fillna(0.0).astype("float64")
    exp["price-mean"] = (pm - pm.mean()) / pm.std()
    assert len(got) == len(exp)
    for c in ("session_id", "item_id-count", "ts-first", "ts-last", "item_id-list", "price-list"):
        _assert_column(got[c], exp[c], c, "list" if c.endswith("list") else None)
    np.testing.assert_allclose(got["price-mean"].to_numpy(), exp["price-mean"].to_numpy(), rtol=1e-5, atol=1e-6)


def test_shuffle_by_keys_keeps_groups_together_and_order(nvt):
    rng = np.random.default_rng(3)
    df = pd.DataFrame({"a": rng.integers(0, 50, 5000), "b": pd.Series([f"v{v}" for v in rng.integers(0, 9, 5000)]),
                       "r": np.arange(5000), "l": [[i, i + 1] for i in range(5000)]})
    ds = nvt.Dataset(df, npartitions=3).shuffle_by_keys(["a", "b"], npartitions=5)
    parts = [p.to_pandas() for p in ds.partitions()]
    assert len(parts) == 5 and sum(len(p) for p in parts) == len(df)
    owner = {}
    for i, p in enumerate(parts):
        assert p["r"].is_monotonic_increasing                 # input order kept
        assert all(list(l) == [r, r + 1] for l, r in zip(p["l"], p["r"]))
        for key in zip(p["a"], p["b"]):
            assert owner.setdefault(key, i) == i


def test_list_slice_workflow_save_reload_in_fresh_process(nvt, tmp_path):
    rng = np.random.default_rng(9)
    df = pd.DataFrame({"y": _ragged(rng, 500, 30)})
    wf = nvt.Workflow(["y"] >> nvt.ops.ListSlice(-5, pad=True, pad_value=1.5))
    first = wf.fit_transform(nvt.Dataset(df)).compute()
    wf.save(str(tmp_path / "wf"))
    df.to_parquet(tmp_path / "in.parquet")
    code = ("import sys, numpy as np, pandas as pd; sys.path.insert(0, %r); import nvtabular as nvt;"
            "wf = nvt.Workflow.load(%r); out = wf.transform(pd.read_parquet(%r));"
            "np.save(%r, np.stack([np.asarray(r, dtype=float) for r in out['y']]))"
            % (ROOT, str(tmp_path / "wf"), str(tmp_path / "in.parquet"), str(tmp_path / "out.npy")))
    subprocess.run([sys.executable, "-c", code], check=True, cwd=str(tmp_path))
    again = np.load(tmp_path / "out.npy")
    np.testing.assert_array_equal(again, np.stack([np.asarray(r, dtype=float) for r in first["y"]]))
