"""CPU tests: operator-graph sugar, column model, dataset partitioning, the C-ABI
library (loads, exports every declared symbol — no compute calls without a GPU),
and the rule that the product never touches the oracle or a CPU fallback."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    from nvtabular_b200 import _build, _lib
    _build.build()
    header = open(os.path.join(ROOT, "include", "nvtb200.h")).read()
    declared = set(re.findall(r"\b(nvtb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed from include/nvtb200.h"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"libnvtb200.so does not export {name}"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    assert _lib.load().nvtb_version() >= 1


def test_library_targets_sm100a_with_256bit_accesses():
    from nvtabular_b200 import _build, _lib
    # the CUDA toolkit that built the library, also when its bin directory is not on PATH
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(_build._nvcc()), "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass or "SM100a" in sass.upper() or "sm_100" in sass
    assert re.search(r"LDG\.E[.\w]*\.256", sass) and re.search(r"STG\.E[.\w]*\.256", sass)


def test_product_never_imports_oracle_or_reference():
    bad = []
    for base, _, files in os.walk(os.path.join(ROOT, "nvtabular_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(base, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "/root/reference" in src:
                    bad.append(os.path.join(base, f))
    assert not bad, bad


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import nvtabular as nvt
    from nvtabular_b200._lib import NvtbError
    df = pd.DataFrame({"a": [1, 2, 2], "x": [1.0, np.nan, 3.0]})
    wf = nvt.Workflow((["a"] >> nvt.ops.Categorify()) + (["x"] >> nvt.ops.FillMissing() >> nvt.ops.Normalize()))
    with pytest.raises(NvtbError):
        wf.fit(nvt.Dataset(df))


def test_column_selector_and_node_sugar():
    import nvtabular as nvt
    from nvtabular import ColumnSelector, ops
    sel = ColumnSelector(["a", ["b", "c"]])
    assert sel.names == ["a", "b", "c"] and sel.grouped_names == ["a", ("b", "c")]
    with pytest.raises(ValueError):
        ColumnSelector([["a", ["b"]]])
    node = ["a", ["b", "c"]] >> ops.Categorify(encode_type="combo")
    assert node.output_columns.names == ["a", "b_c"]
    joint = [["b", "c"]] >> ops.Categorify()
    assert joint.output_columns.names == ["b", "c"]
    conts = ["x", "y"] >> ops.FillMissing(add_binary_cols=True) >> ops.Normalize()
    assert conts.output_columns.names == ["x", "y", "x_filled", "y_filled"]
    both = node + conts + "label"
    assert both.output_columns.names == ["a", "b_c", "x", "y", "x_filled", "y_filled", "label"]
    assert (both - ["label"]).output_columns.names == ["a", "b_c", "x", "y", "x_filled", "y_filled"]
    assert both[["a", "x"]].output_columns.names == ["a", "x"]
    assert nvt.Workflow(both).output_node.root_columns() == ["a", "b", "c", "x", "y", "label"]
    as_class = ["a"] >> ops.Categorify          # ops may be passed as classes
    assert isinstance(as_class.op, ops.Categorify)
    jg = ["u", ["u", "m"]] >> ops.JoinGroupby(cont_cols=["r"], stats=["count", "sum"])
    assert jg.output_columns.names == ["u_count", "u_r_sum", "u_m_count", "u_m_r_sum"]
    te = ["u", ["u", "m"]] >> ops.TargetEncoding("r", kfold=3, drop_folds=False)
    assert te.output_columns.names == ["TE_u_r", "TE_u_m_r", "__fold__"]
    with pytest.raises(ValueError):
        ops.JoinGroupby(cont_cols=["r"], stats=["median"])
    with pytest.raises(TypeError):
        ops.HashBucket("ten")


def test_categorify_kwarg_validation():
    from nvtabular import ops
    for bad in (dict(start_index=1), dict(na_sentinel=0), dict(bogus=1), dict(encode_type="x"),
                dict(num_buckets=0), dict(freq_threshold=1, max_size=5), dict(search_sorted=True, freq_threshold=2),
                dict(encode_type="combo", vocabs={"a": pd.Series([1])}), dict(num_buckets=1.5), dict(max_size="3")):
        with pytest.raises(ValueError):
            ops.Categorify(**bad)
    with pytest.warns(UserWarning):
        ops.Categorify(num_buckets=10)
    with pytest.warns(FutureWarning):
        ops.Categorify(tree_width=4)
    assert ops.Categorify().output_dtype == np.int64 and ops.Categorify(dtype=np.int32).output_dtype == np.int32
    assert ops.emb_sz_rule(29) == (29, 16)


def test_column_roundtrip_and_bitmask():
    from nvtabular_b200.column import Column, DeviceFrame, pack_validity, unpack_validity
    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 255, 1000):
        v = torch.from_numpy(rng.random(n) < 0.5)
        m = pack_validity(v)
        assert m.numel() % 32 == 0 and torch.equal(unpack_validity(m, n), v)
        if n:   # Arrow layout: bit (i & 7) of byte (i >> 3)
            i = n - 1
            assert bool((int(m[i >> 3]) >> (i & 7)) & 1) == bool(v[i])
    df = pd.DataFrame({
        "i": pd.array([1, None, 3], dtype="Int32"), "f": [1.5, np.nan, 2.5], "s": ["b", None, "a"],
        "l": [[1, 2], [], [3]], "b": [True, False, True], "u": np.array([1, 2, 3], dtype="uint16"),
    })
    fr = DeviceFrame.from_pandas(df, device="cpu")
    assert fr["i"].data.dtype == torch.int32 and fr["i"].null_count() == 1
    assert fr["s"].dictionary.tolist() == ["a", "b"] and fr["s"].data.tolist()[0] == 1
    assert fr["l"].offsets.tolist() == [0, 2, 2, 3] and fr["u"].data.dtype == torch.int32
    back = pd.DataFrame({k: c.to_pandas(k) for k, c in fr.items()})
    assert back["i"].tolist()[0] == 1 and np.isnan(back["i"].tolist()[1])
    assert back["s"].tolist()[0] == "b" and back["s"].isna().tolist() == [False, True, False]
    assert [list(x) for x in back["l"]] == [[1, 2], [], [3]] and back["b"].tolist() == [True, False, True]


def test_dataset_partitions_like_dask_from_pandas():
    import nvtabular as nvt
    df = pd.DataFrame({"a": np.arange(26)})
    ds = nvt.Dataset(df, npartitions=3, device="cpu")
    assert [len(p) for p in ds.partitions()] == [9, 9, 8]
    assert ds.num_rows == 26 and ds.schema.column_names == ["a"]
    assert ds.to_ddf().compute()["a"].tolist() == list(range(26))


def test_keyspace_string_and_float_keys_are_order_preserving():
    from nvtabular_b200.column import Column
    from nvtabular_b200.ops.keyspace import KeySpace, _float_to_key, _key_to_float
    a = Column.from_strings(["pear", "apple", None, "fig"], device="cpu")
    b = Column.from_strings(["kiwi", "apple"], device="cpu")
    ks = KeySpace.for_columns([a, b])
    assert ks.dictionary.tolist() == ["apple", "fig", "kiwi", "pear"]
    assert ks.keys_for(a).data.tolist() == [3, 0, 0, 1] and ks.keys_for(b).data.tolist() == [2, 0]
    unseen = Column.from_strings(["zzz", "apple", "aaa"], device="cpu")
    k = ks.keys_for(unseen).data.tolist()
    assert k[1] == 0 and k[0] < 0 and k[2] < 0 and k[0] != k[2]
    assert ks.decode(np.array([0, 3])).tolist() == ["apple", "pear"]
    x = np.array([-1e300, -2.5, -0.0, 0.0, 1e-300, 3.0, np.inf])
    key = _float_to_key(Column(torch.from_numpy(x))).data.numpy()
    assert (np.diff(key) >= 0).all() and key[2] == key[3]
    np.testing.assert_array_equal(_key_to_float(key), np.where(x == 0, 0.0, x))


def test_fold_hash_is_a_bijection_with_the_documented_inverse():
    """csrc/common.cuh fold_hash / fold_unhash: the shared-memory tables of the group-by and
    the encode store h = fold_hash(key) and recover the key with the inverse.  The constants
    are read from the header; the arithmetic is restated here."""
    src = open(os.path.join(ROOT, "nvtabular_b200", "csrc", "common.cuh")).read()
    c = {k: int(v, 16) for k, v in re.findall(r"constexpr uint32_t (kFold\w+) = (0x[0-9A-Fa-f]+)u;", src)}
    M = 0xFFFFFFFF
    assert (c["kFoldC1"] * c["kFoldC1Inv"]) & M == 1 and (c["kFoldC2"] * c["kFoldC2Inv"]) & M == 1
    assert c["kFoldC1"] & 1 and c["kFoldC2"] & 1

    def fold_hash(k):
        h = (k * c["kFoldC1"]) & M
        h ^= h >> 15
        return (h * c["kFoldC2"]) & M

    def fold_unhash(h):
        h = (h * c["kFoldC2Inv"]) & M
        h ^= h >> 15
        h ^= h >> 30
        return (h * c["kFoldC1Inv"]) & M

    rng = np.random.default_rng(3)
    keys = [0, 1, M, 0x80000000, 0x7FFFFFFF] + [int(x) for x in rng.integers(0, 1 << 32, 20000)]
    hs = [fold_hash(k) for k in keys]
    assert [fold_unhash(h) for h in hs] == keys
    assert len(set(hs)) == len(set(keys))
    # exactly one key maps to the value the shared tables reserve for "empty"
    assert fold_hash(fold_unhash(c["kFoldEmpty"])) == c["kFoldEmpty"]
    # the partition digit (top bits) spreads sequential ids: no partition of 1024 gets > 2x its share
    top = np.bincount([fold_hash(k) >> 22 for k in range(200000)], minlength=1024)
    assert top.max() < 2 * 200000 / 1024


def test_workflow_fits_host_blocking_ops_first(monkeypatch):
    """ops of one phase are independent; the ones whose fit ends in a blocking device->host read
    (Normalize's moments) are fitted first so that the read does not drain Categorify's queue"""
    import nvtabular_b200 as nvt
    from nvtabular_b200 import ops
    order = []
    for cls in (ops.Categorify, ops.Normalize):
        monkeypatch.setattr(cls, "fit", lambda self, cols, ddf, _n=cls.__name__: order.append(_n) or {})
        monkeypatch.setattr(cls, "fit_finalize", lambda self, stats: None)
    monkeypatch.setattr(nvt.Workflow, "fit_schema", lambda self, schema: self)
    wf = nvt.Workflow((["c"] >> ops.Categorify()) + (["x"] >> ops.FillMissing() >> ops.Normalize()))

    class _DS:
        schema = None
    wf.fit(_DS())
    assert order == ["Normalize", "Categorify"]


def test_bench_clock_sampler_window():
    """bench.py keeps the nvidia-smi samples whose own timestamps fall inside the timed region"""
    sys.path.insert(0, ROOT)
    import bench
    import datetime
    t = datetime.datetime(2026, 1, 2, 3, 4, 5, 250000)
    assert abs(bench.ClockSampler._epoch(t.strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]) - t.timestamp()) < 1e-3
    assert bench.ClockSampler._epoch("garbage") is None


def _frames_equal(a: pd.DataFrame, b: pd.DataFrame):
    assert list(a.columns) == list(b.columns) and len(a) == len(b)
    for c in a.columns:
        x, y = a[c], b[c]
        if not (pd.api.types.is_numeric_dtype(x.dtype) and pd.api.types.is_numeric_dtype(y.dtype)):
            for u, v in zip(x.tolist(), y.tolist()):
                if isinstance(u, (list, np.ndarray)) or isinstance(v, (list, np.ndarray)):
                    assert list(u) == list(v)
                else:
                    assert (u == v) or (pd.isna(u) and pd.isna(v))
        else:
            np.testing.assert_array_equal(np.asarray(x, dtype="float64"), np.asarray(y, dtype="float64"))


def test_arrow_ingest_keeps_nullable_ints_and_the_bitmask(tmp_path):
    """Column.from_arrow: data buffer + Arrow validity bitmap map 1:1 onto (data, validity);
    nullable int32 stays int32 (pandas would make it float64), sliced arrays with a bit offset
    that is not byte aligned are repacked, bools/strings/lists/dictionaries go through."""
    import pyarrow as pa
    from nvtabular_b200.column import Column, DeviceFrame, unpack_validity
    rng = np.random.default_rng(0)
    n = 1003
    vals = rng.integers(-5, 5, n).astype("int32")
    mask = rng.random(n) < 0.3
    arr = pa.array(vals, mask=mask)
    for a in (arr, arr.slice(8, 500), arr.slice(3, 77), pa.chunked_array([arr.slice(0, 10), arr.slice(10)])):
        col = Column.from_arrow(a, torch.device("cpu"))
        py = a.to_pylist()
        assert col.data.dtype == torch.int32 and len(col) == len(py)
        valid = unpack_validity(col.validity, len(py)).numpy()
        np.testing.assert_array_equal(valid, np.array([v is not None for v in py]))
        np.testing.assert_array_equal(col.data.numpy()[valid], np.array([v for v in py if v is not None], dtype="int32"))
        assert col.validity.numel() % 32 == 0
        # the round trip back to arrow is exact
        assert col.to_arrow().to_pylist() == py
    assert Column.from_arrow(pa.array(vals), torch.device("cpu")).validity is None
    b = Column.from_arrow(pa.array([True, None, False]), torch.device("cpu"))
    assert b.is_bool and b.to_arrow().to_pylist() == [True, None, False]
    s = Column.from_arrow(pa.array(["b", None, "a", "b"]).dictionary_encode(), torch.device("cpu"))
    sp = s.to_pandas().tolist()
    assert s.is_string and sp[0] == "b" and pd.isna(sp[1]) and sp[2:] == ["a", "b"]
    assert s.data.tolist()[0] > s.data.tolist()[2]          # order-preserving codes
    li = Column.from_arrow(pa.array([[1, 2], [], None, [3]], type=pa.list_(pa.int64())), torch.device("cpu"))
    assert li.is_list and li.offsets.tolist() == [0, 2, 2, 2, 3] and li.data.tolist() == [1, 2, 3]
    small = Column.from_arrow(pa.array([1, 2, 3], type=pa.int8()), torch.device("cpu"))
    assert small.data.dtype == torch.int32


def test_parquet_dataset_roundtrip_without_pandas_upcast(tmp_path):
    """Dataset(path.parquet): one partition per row group (or per part_size rows), nullable
    int32 columns arrive as int32 + bitmask; to_parquet writes what compute() shows."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    import nvtabular_b200 as nvt
    rng = np.random.default_rng(1)
    n = 5000
    tbl = pa.table({
        "C1": pa.array(rng.integers(0, 50, n).astype("int32"), mask=rng.random(n) < 0.1),
        "I1": pa.array(rng.integers(-3, 1000, n).astype("int32"), mask=rng.random(n) < 0.4),
        "x": pa.array(rng.normal(size=n)),
        "s": pa.array(rng.choice(["u", "v", "w"], n)),
    })
    path = str(tmp_path / "in.parquet")
    pq.write_table(tbl, path, row_group_size=1200)
    ds = nvt.Dataset(path, engine="parquet", device=torch.device("cpu"))
    assert ds.npartitions == 5
    parts = list(ds.partitions())
    assert parts[0]["C1"].data.dtype == torch.int32 and parts[0]["C1"].validity is not None
    assert ds.schema["I1"].dtype == np.dtype("int32")
    got = ds.to_ddf().compute()
    _frames_equal(got, tbl.to_pandas())
    # part_size in rows regroups row groups; a directory of part files is read in name order
    ds2 = nvt.Dataset(path, part_size=2048, device=torch.device("cpu"))
    assert [len(p) for p in ds2.partitions()] == [2048, 2048, 904]
    out_dir = str(tmp_path / "out")
    ds2.to_parquet(out_dir)
    back = nvt.Dataset(out_dir, device=torch.device("cpu"))
    assert back.npartitions == 3
    _frames_equal(back.to_ddf().compute(), tbl.to_pandas())
    assert pq.read_table(os.path.join(out_dir, "part_0.parquet")).schema.field("C1").type == pa.int32()


# ------------------------------------------------------------------ round 2: artefact + save/load host logic
def test_fast_parquet_writer_roundtrips_like_pandas(tmp_path):
    """unique.<col>.parquet is written with pyarrow directly (no pandas conversion, no dictionary
    pages); pandas must read back exactly what DataFrame.to_parquet would have produced: the
    RangeIndex that carries the labels (categorify.py:745-760) and the column dtypes."""
    import numpy as np
    import pandas as pd
    from nvtabular_b200.ops.categorify import _write_numeric_parquet
    keys = np.array([40, 7, 19, -3], dtype=np.int32)
    sizes = np.array([9, 4, 4, 1], dtype=np.int64)
    _write_numeric_parquet(str(tmp_path / "unique.C1.parquet"), {"C1": keys, "C1_size": sizes}, index_start=3)
    got = pd.read_parquet(tmp_path / "unique.C1.parquet")
    exp = pd.DataFrame({"C1": keys, "C1_size": sizes})
    exp.index = pd.RangeIndex(3, 7)
    pd.testing.assert_frame_equal(got, exp)
    assert isinstance(got.index, pd.RangeIndex) and got.index.start == 3


def test_stat_file_key_columns_keep_their_dtype_with_a_null_row(tmp_path):
    """cat_stats files carry the null group as a null KEY: int keys must come back as (nullable)
    ints, not float64 — a reloaded table otherwise sits in another key space than the column"""
    import numpy as np
    import pandas as pd
    from nvtabular_b200.ops._tables import key_columns
    from nvtabular_b200.ops.keyspace import KeySpace
    cols = key_columns(KeySpace("int", None, np.dtype("int32")), ["u"], np.array([5, 3, 9]), with_null_row=True)
    df = pd.DataFrame(cols)
    df["u_count"] = [2, 1, 1, 0]
    df.to_parquet(tmp_path / "cat_stats.u.parquet")
    back = pd.read_parquet(tmp_path / "cat_stats.u.parquet")
    assert str(back["u"].dtype) == "Int32" and back["u"].isna().tolist() == [False, False, False, True]
    assert back["u"].dropna().astype("int32").tolist() == [5, 3, 9]
    fl = key_columns(KeySpace("float", None, np.dtype("float64")), ["x"],
                     np.array([0, 4607182418800017408], dtype=np.int64), with_null_row=True)   # keys of 0.0, 1.0
    assert fl["x"].dtype == np.float64 and np.isnan(fl["x"].iloc[-1])


def test_graph_json_roundtrip_of_stateless_and_float_state_ops(tmp_path):
    """Workflow.save / Workflow.load (reference layout: workflow.py:256-348, graph_serializer.py:
    1077-1165) for the operators whose fitted state is plain floats — no device needed: DAG shape,
    selectors with multi-column groups, operator parameters and the restored statistics."""
    import json
    import nvtabular_b200 as nvt
    ops = nvt.ops
    norm = ops.Normalize(out_dtype="float32")
    norm.means, norm.stds = {"x": 1.5, "y": -2.0}, {"x": 0.5, "y": 4.0}
    mm = ops.NormalizeMinMax()
    mm.mins, mm.maxs = {"z": 0.0}, {"z": 10.0}
    graph = (["x", "y"] >> ops.FillMissing(fill_val=7) >> norm) + (["z"] >> mm) + \
        (["w"] >> ops.Clip(min_value=0, max_value=9) >> ops.LogOp()) + (["k"] >> ops.HashBucket(13)) + ["label"]
    wf = nvt.Workflow(graph)
    wf.save(str(tmp_path / "wf"))
    meta = json.load(open(tmp_path / "wf" / "metadata.json"))
    assert "nvtabular" in meta["versions"] and "generated_timestamp" in meta
    g = json.load(open(tmp_path / "wf" / "graph.json"))
    assert g["format_version"] == 1
    by_class = {}
    for n in g["nodes"]:
        by_class.setdefault(n["op_class"], []).append(n)
    assert by_class["nvtabular.ops.normalize.Normalize"][0]["op_state"]["means"] == {"x": 1.5, "y": -2.0}
    assert by_class["nvtabular.ops.clip.Clip"][0]["op_params"] == {"min_value": 0, "max_value": 9}
    assert "merlin.dag.ops.concat_columns.ConcatColumns" in by_class and "merlin.dag.ops.selection.SelectionOp" in by_class
    ids = {n["id"] for n in g["nodes"]}
    assert all(set(n["parent_ids"]) <= ids for n in g["nodes"]) and g["output_node_id"] in ids
    wf2 = nvt.Workflow.load(str(tmp_path / "wf"))
    order = wf2.output_node.topo_order()
    kinds = [n.kind for n in order]
    assert kinds.count("input") == 5 and kinds.count("concat") >= 1
    ops2 = {type(n.op).__name__: n.op for n in order if n.kind == "op"}
    assert ops2["Normalize"].means == {"x": 1.5, "y": -2.0} and ops2["Normalize"].stds == {"x": 0.5, "y": 4.0}
    assert str(ops2["Normalize"].out_dtype) == "float32"
    assert ops2["NormalizeMinMax"].maxs == {"z": 10.0} and ops2["FillMissing"].fill_val == 7
    assert ops2["Clip"].min_value == 0 and ops2["Clip"].max_value == 9 and ops2["HashBucket"].num_buckets == 13
    assert sorted(wf2.output_node.output_columns.names) == ["k", "label", "w", "x", "y", "z"]
    with pytest.raises(nvt.serialize.WorkflowSerializationError):
        bad = dict(g)
        bad["format_version"] = 99
        json.dump(bad, open(tmp_path / "wf" / "graph.json", "w"))
        nvt.Workflow.load(str(tmp_path / "wf"))


def test_operator_hooks_without_device():
    """compute_selector / supported_formats / inference_initialize contracts (categorify.py:589-609)"""
    import warnings
    import nvtabular_b200 as nvt
    from nvtabular_b200.graph import ColumnSchema, Schema
    from nvtabular_b200.inference import DataFormats
    op = nvt.ops.Normalize()
    sel = nvt.ColumnSelector(["a", "b"])
    assert op.compute_selector(Schema([ColumnSchema("a"), ColumnSchema("b")]), sel, sel, None) is sel
    with pytest.raises(ValueError):
        op.compute_selector(Schema([ColumnSchema("a")]), sel, sel, None)
    assert op.supported_formats & DataFormats.NUMPY_DICT_ARRAY and op.supported_formats & DataFormats.PANDAS_DATAFRAME
    assert nvt.ops.HashBucket(3).supported_formats & DataFormats.PANDAS_DATAFRAME
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert nvt.ops.Categorify(encode_type="combo").inference_initialize(sel, {}) is None
        assert any("combo" in str(x.message) for x in w)
    assert nvt.ops.FillMissing(add_binary_cols=True).inference_initialize(sel, {}) is None


def test_reference_arm_under_torchrun_prints_one_line(tmp_path):
    """The driver launches `bench.py --impl reference --gpus N` the way it launches the GPU arm
    (torchrun, N ranks): rank 0 alone runs the CPU path and prints ONE JSON line with the contract's
    keys; the other ranks exit 0 without work."""
    import json
    port = 29700 + os.getpid() % 200
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "bench.py"),
           "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-rows", "60000"]
    env = dict(os.environ, NVTB_REF_BUDGET_S="20")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 1 and d["higher_is_better"] is True
    assert d["unit"] == "rows/s" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "cpu_model" in d["cpu_baseline"]
    assert d["config"]["total_rows"] == 2 * d["config"]["rows_per_gpu"] and "configs[2]" in d["config"]["workload"]


def test_bench_e2e_rows_fit_the_host_memory_limit():
    """bench.py sizes the pinned e2e leg to the container's memory limit: unchanged where the known
    boxes have room (200 GiB for 1 GPU, 137 GB per GPU beyond), whole 2^23-row partitions and never
    zero where they do not."""
    import bench
    G = 1 << 30
    want, bpr = 1 << 27, bench.E2E_PINNED_BYTES_PER_ROW
    assert bench.e2e_rows_within_host_memory(want, bpr, 1, 200 * G) == want
    assert bench.e2e_rows_within_host_memory(want, bpr, 2, 256 * G) == want
    assert bench.e2e_rows_within_host_memory(want, bpr, 8, 1024 * G) == want
    assert bench.e2e_rows_within_host_memory(want, bpr, 1, None) == want
    small = bench.e2e_rows_within_host_memory(want, bpr, 8, 200 * G)
    assert small % (1 << 23) == 0 and 0 < small < want
    assert 8 * small * bpr <= 0.8 * 200 * G
    assert bench.e2e_rows_within_host_memory(want, bpr, 8, 1 * G) == 1 << 23
    b = bench._host_memory_budget()
    assert b is None or b > 0


def test_bench_output_sample_gathers_the_same_rows_of_every_partition(tmp_path):
    """bench.py --dump-outputs: one seeded sample of rows across uneven partitions, integers as exact
    float64, float32 kept, nulls of a bitmask column as NaN, the same rows from run to run"""
    import bench
    from nvtabular_b200.column import Column, DeviceFrame, pack_validity
    rng = np.random.default_rng(1)
    n = 300_007
    full = {"a": rng.integers(0, 1 << 40, n), "x": rng.standard_normal(n).astype(np.float32),
            "i": rng.integers(-5, 5, n).astype(np.int32)}
    valid = rng.random(n) < 0.7
    frame = DeviceFrame({"a": Column(torch.from_numpy(full["a"])), "x": Column(torch.from_numpy(full["x"])),
                         "i": Column(torch.from_numpy(full["i"]), pack_validity(torch.from_numpy(valid)))})
    parts = bench.cut(frame, 3)
    sample = bench.OutputSample([len(p) for p in parts], 3, "cpu")
    for i, p in enumerate(parts):
        sample.take(i, p)
    names, nbytes = sample.save(str(tmp_path))
    assert names == ["a", "i", "row_index", "x"] and nbytes <= bench.DUMP_BYTES
    row = np.load(tmp_path / "row_index.npy")
    assert row.dtype == np.float64 and len(row) == bench.DUMP_ROWS and (np.diff(row) > 0).all()
    row = row.astype(np.int64)
    np.testing.assert_array_equal(row, bench.OutputSample([len(p) for p in parts], 3, "cpu").rows)
    a, x, i = (np.load(tmp_path / f"{c}.npy") for c in ("a", "x", "i"))
    assert a.dtype == np.float64 and x.dtype == np.float32 and i.dtype == np.float64
    np.testing.assert_array_equal(a, full["a"][row].astype(np.float64))
    np.testing.assert_array_equal(x, full["x"][row])
    np.testing.assert_array_equal(i, np.where(valid[row], full["i"][row], np.nan))


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs writes every output column of its timed step at the seeded sample
    rows; a fit + transform of the same table in this process gives the same values"""
    import json
    import bench
    import nvtabular_b200 as nvt
    rows, parts, profile = 1 << 20, 3, 40_000_000
    dump = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(rows), "--parts", str(parts),
           "--profile-rows", str(profile), "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu-baseline",
           "--no-gate", "--dump-outputs", str(dump)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    wf = bench.build_workflow(nvt, "criteo", str(tmp_path / "wf"))
    names = wf.output_node.output_columns.names
    assert sorted(os.listdir(dump)) == sorted(n + ".npy" for n in names + ["row_index"])
    assert sum(os.path.getsize(dump / f) for f in os.listdir(dump)) <= bench.DUMP_BYTES
    row = np.load(dump / "row_index.npy").astype(np.int64)
    table = bench.make_table("criteo", rows, torch.device("cuda"), 0, profile)
    wf.fit(nvt.Dataset(bench.cut(table, parts)))
    out = wf.transform(table)
    for c in names:
        got = np.load(dump / f"{c}.npy")
        exp = out[c].data[torch.from_numpy(row).cuda()].cpu().numpy()
        assert len(got) == len(row) and not np.isnan(got).any(), c
        if exp.dtype.kind in "iu":
            np.testing.assert_array_equal(got, exp.astype(np.float64), err_msg=c)
        else:
            np.testing.assert_allclose(got, exp, rtol=1e-9, atol=1e-12, err_msg=c)
