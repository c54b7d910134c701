"""Session ops without a GPU: the reference's ListSlice and Groupby known-answer tests
(tests/unit/ops/test_list_slice.py, tests/unit/ops/test_groupyby.py) re-typed against the oracle,
the operators' schemas through Workflow.fit_schema, argument checks, graph.json records, and the
row-count check of frames merged by the workflow."""
import json

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import sessions as osess

Y = [[0, 1, 2, 2, 767], [1, 2, 2, 3], [1, 223, 4]]


# reference tests/unit/ops/test_list_slice.py::test_list_slice
@pytest.mark.parametrize("args,expected", [
    ((0, 2), [[0, 1], [1, 2], [1, 223]]),
    ((3, 5), [[2, 767], [3], []]),
    ((4, 10), [[767], [], []]),
    ((100, 20000), [[], [], []]),
    ((-4,), [[1, 2, 2, 767], [1, 2, 2, 3], [1, 223, 4]]),
    ((-3, -1), [[2, 2], [2, 2], [1, 223]]),
])
def test_list_slice_kat(args, expected):
    assert osess.list_slice(Y, *args) == expected


# reference tests/unit/ops/test_list_slice.py::test_list_slice_pad
@pytest.mark.parametrize("args,kw,expected", [
    ((5,), {}, [[0, 1, 2, 2, 767], [1, 2, 2, 3, 0], [1, 223, 4, 0, 0]]),
    ((1, 6), {"pad_value": 123}, [[1, 2, 2, 767, 123], [2, 2, 3, 123, 123], [223, 4, 123, 123, 123]]),
    ((-4,), {"pad_value": -1}, [[1, 2, 2, 767], [1, 2, 2, 3], [1, 223, 4, -1]]),
    ((-4, -1), {"pad_value": -1}, [[1, 2, 2], [1, 2, 2], [1, 223, -1]]),
])
def test_list_slice_pad_kat(args, kw, expected):
    assert osess.list_slice(Y, *args, pad=True, **kw) == expected


def _timeseries(seed, size=60):
    """the frame of reference test_groupyby.py::test_groupby_op"""
    rng = np.random.default_rng(seed)
    df = pd.DataFrame({"name": rng.choice(["Dave", "Zelda"], size=size), "id": rng.choice([0, 1], size=size),
                       "ts": np.linspace(0.0, 10.0, num=size), "x": np.arange(size),
                       "y": np.linspace(0.0, 10.0, num=size), "shuffle": rng.uniform(0.0, 10.0, size=size)})
    return df.sort_values("shuffle").drop(columns="shuffle").reset_index(drop=True)


# reference tests/unit/ops/test_groupyby.py::test_groupby_op (the invariants it checks)
@pytest.mark.parametrize("keys", [["name"], "id", ["name", "id"]])
@pytest.mark.parametrize("ascending", [True, False])
def test_groupby_invariants(keys, ascending):
    df = _timeseries(0)
    out = osess.groupby(df, keys, ["ts"], {"x": ["list", "sum", "first", "last"], "y": ["first", "last"],
                                           "ts": ["min"]}, name_sep="-", ascending=ascending)
    for i, el in enumerate(out["x-list"]):
        s = pd.Series(el)
        assert s.is_monotonic_increasing if ascending else s.is_monotonic_decreasing
        assert out["x-sum"].iloc[i] == s.sum()
        assert out["x-first"].iloc[i] == (el[0] if ascending else el[-1])
    assert (out["y-first"] < out["y-last"]).all()


# reference tests/unit/ops/test_groupyby.py::test_groupby_casting_in_aggregations
def test_groupby_casting_in_aggregations():
    rng = np.random.default_rng(1)
    df = pd.DataFrame({"name": rng.choice(["Dave", "Zelda"], size=60), "x": rng.integers(0, 2, 60).astype(np.int8),
                       "y": np.linspace(0.0, 10.0, 60), "z": np.linspace(0.0, 10.0, 60).astype(np.float32)})
    aggs = ["mean", "std", "var", "median", "nunique", "sum"]
    out = osess.groupby(df, "name", None, {c: aggs for c in "xyz"}, name_sep="-")
    ref = df.set_index("name")
    for agg in aggs:
        for col in "xyz":
            for name in ("Dave", "Zelda"):
                want = getattr(ref.loc[name][col], agg)()
                assert np.allclose(want, out.loc[out.name == name, f"{col}-{agg}"].item())
                assert out[f"{col}-{agg}"].dtype == (np.int32 if agg == "nunique" else np.float32)


@pytest.fixture(scope="module")
def nvt():
    import nvtabular
    return nvtabular


def _fit_schema(nvt, node, names, **schemas):
    cols = [schemas.get(n) or nvt.ColumnSchema(n) for n in names]
    return nvt.Workflow(node).fit_schema(nvt.Schema(cols))


# reference tests/unit/ops/test_groupyby.py::test_groupby_selector_cols
def test_groupby_schema_selector_names_dtypes_tags(nvt):
    from nvtabular_b200.graph import ColumnSchema
    aggs = {"x": ["list", "sum", "count"], "y": ["first", "last", "median", "nunique"], "ts": ["min"]}
    x = ColumnSchema("x", np.dtype("int64"), tags=["custom_tag"])
    ts = ColumnSchema("ts", np.dtype("float64"))
    wf = _fit_schema(nvt, ["name", "id", "ts", "x", "y"] >> nvt.ops.Groupby(
        groupby_cols=["name"], sort_cols=["ts"], aggs=aggs, name_sep="-"), ["name", "id", "ts", "x", "y"], x=x, ts=ts)
    schema = wf.output_schema
    assert schema.column_names == ["name", "x-list", "x-sum", "x-count", "y-first", "y-last", "y-median",
                                   "y-nunique", "ts-min"]
    assert schema["x-list"].is_list and schema["x-list"].is_ragged and schema["x-list"].dtype == np.dtype("int64")
    assert "custom_tag" in schema["x-list"].tags
    assert schema["x-sum"].dtype == np.float32 and schema["x-count"].dtype == np.int32
    assert schema["y-median"].dtype == np.float32 and schema["y-nunique"].dtype == np.int32
    assert schema["ts-min"].dtype == np.dtype("float64") and not schema["ts-min"].is_list
    wf = _fit_schema(nvt, ["id", "ts", "x", "y"] >> nvt.ops.Groupby(
        groupby_cols=["name"], sort_cols=["ts"], aggs=aggs, name_sep="-"), ["name", "id", "ts", "x", "y"])
    assert "name" not in wf.output_schema.column_names
    # reference test_groupby_without_selector_in_groupby_cols; "__all__" and the builtin `list`
    node = ["product_id"] >> nvt.ops.Groupby(groupby_cols=["day"], aggs="count")
    assert node.output_columns.names == ["product_id_count"]
    assert node.dependencies[0].output_columns.names == ["day"]
    node = ["day", "a", "b"] >> nvt.ops.Groupby(groupby_cols="day", aggs=[list, "max"])
    assert node.output_columns.names == ["day", "a_list", "a_max", "b_list", "b_max"]


def test_groupby_rejects_bad_aggs(nvt):
    from nvtabular_b200.graph import ColumnSchema
    with pytest.raises(ValueError):
        nvt.ops.Groupby(groupby_cols="k", aggs={"x": "mode"})
    lst = ColumnSchema("l", np.dtype("int64"), is_list=True, is_ragged=True)
    with pytest.raises(ValueError, match="nested"):
        _fit_schema(nvt, ["k", "l"] >> nvt.ops.Groupby(groupby_cols="k", aggs={"l": "list"}), ["k", "l"], l=lst)
    wf = _fit_schema(nvt, ["k", "l"] >> nvt.ops.Groupby(groupby_cols="k", aggs={"l": ["first", "last"]}),
                     ["k", "l"], l=lst)
    assert wf.output_schema["l_first"].is_list
    s = ColumnSchema("s", np.dtype("O"))
    for agg in ("sum", "mean", "std", "var", "median"):
        with pytest.raises(TypeError, match="string"):
            _fit_schema(nvt, ["k", "s"] >> nvt.ops.Groupby(groupby_cols="k", aggs={"s": agg}), ["k", "s"], s=s)
    wf = _fit_schema(nvt, ["k", "s"] >> nvt.ops.Groupby(groupby_cols="k", aggs={"s": ["count", "nunique", "max"]}),
                     ["k", "s"], s=s)
    assert wf.output_schema["s_max"].dtype == np.dtype("O")


def test_list_slice_schema_and_bounds(nvt):
    from nvtabular_b200.graph import ColumnSchema, Tags
    y = ColumnSchema("y", np.dtype("int64"), is_list=True, is_ragged=True)
    for op, vc in ((nvt.ops.ListSlice(0, 20), {"min": 0, "max": 20}), (nvt.ops.ListSlice(-20, pad=True),
                                                                       {"min": 20, "max": 20}),
                   (nvt.ops.ListSlice(2), {"min": 0, "max": 2}), (nvt.ops.ListSlice(1, None), {"min": 0, "max": 1}),
                   (nvt.ops.ListSlice(0), {"min": 0, "max": None}), (nvt.ops.ListSlice(-3, -1), {"min": 0, "max": 2})):
        cs = _fit_schema(nvt, ["y"] >> op, ["y"], y=y).output_schema["y"]
        assert cs.properties["value_count"] == vc and Tags.LIST in cs.tags and cs.is_list
        assert cs.dtype == np.dtype("int64")
        assert op.max_elements == osess.list_slice_bounds(*((op.start, op.end)))[2]
    for bad in ((0,), (-3, 5), (2, -1), (3, 1)):
        if bad == (-3, 5):
            assert nvt.ops.ListSlice(*bad, pad=True).max_elements == 3
            continue
        with pytest.raises(ValueError):
            nvt.ops.ListSlice(*bad, pad=True)


def test_list_slice_graph_json_and_groupby_save_refused(nvt, tmp_path):
    from nvtabular_b200.graph import ColumnSchema
    y = ColumnSchema("y", np.dtype("float32"), is_list=True, is_ragged=True)
    wf = _fit_schema(nvt, ["y"] >> nvt.ops.ListSlice(-5, pad=True, pad_value=2.5), ["y"], y=y)
    wf.save(str(tmp_path / "ls"))
    graph = json.load(open(tmp_path / "ls" / "graph.json"))
    rec = [r for r in graph["nodes"] if r["op_class"].endswith("ListSlice")]
    assert len(rec) == 1 and rec[0]["op_class"] == "nvtabular.ops.list_slice.ListSlice"
    assert rec[0]["op_params"] == {"start": -5, "end": int(np.iinfo(np.int64).max), "pad": True, "pad_value": 2.5}
    back = nvt.Workflow.load(str(tmp_path / "ls"))
    op = back.output_node.op
    assert (op.start, op.end, op.pad, op.pad_value, op.max_elements) == (-5, np.iinfo(np.int64).max, True, 2.5, 5)

    gb = _fit_schema(nvt, ["k", "x"] >> nvt.ops.Groupby(groupby_cols="k"), ["k", "x"])
    with pytest.raises(NotImplementedError, match="Groupby"):
        gb.save(str(tmp_path / "gb"))


def test_merged_frames_must_have_equal_row_counts(nvt):
    from nvtabular_b200.column import Column, DeviceFrame
    from nvtabular_b200.ops.base import Operator

    class Halve(Operator):          # stands in for a row-count-changing op such as Groupby
        def transform(self, col_selector, df):
            return DeviceFrame({n: Column(df[n].data[: len(df) // 2]) for n in col_selector.names})

    frame = DeviceFrame({"a": Column(torch.arange(10)), "b": Column(torch.arange(10))})
    ok = nvt.Workflow((["a"] >> Halve()) + (["b"] >> Halve()))
    assert len(ok.transform(frame)) == 5
    bad = nvt.Workflow((["a"] >> Halve()) + ["b"])
    with pytest.raises(ValueError, match="different row counts"):
        bad.transform(frame)
    dep = nvt.Workflow(["b"] >> Halve() >> Halve())
    assert len(dep.transform(frame)) == 2
