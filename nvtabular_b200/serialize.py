"""Workflow.save / Workflow.load in the reference's on-disk layout
(nvtabular/workflow/workflow.py:256-348, nvtabular/workflow/graph_serializer.py:16-29, 985-1165):

    saved_workflow/
      metadata.json            versions + timestamp
      graph.json               {"format_version": 1, "output_node_id", "nodes": [...]}: per node
                               id, op_class, op_params, op_state, parent_ids, dependency_ids,
                               selector, input_schema, output_schema
      artifacts/node_<id>/     file-based fitted state of one operator
        categories/unique.<col>.parquet, meta.<col>.parquet, cat_stats.<name>.parquet

No pickle.  Operator classes are recorded under the reference's module paths
(`nvtabular.ops.categorify.Categorify`, ...) and the graph plumbing under merlin's
(`merlin.dag.ops.selection.SelectionOp`, `...concat_columns.ConcatColumns`,
`...subtraction.SubtractionOp`, `...subset_columns.SubsetColumns`), so that the files describe
the same DAG to either implementation.  Fitted state that lives in HBM here (vocabulary lookups,
group tables) is rebuilt lazily from the parquet artefacts after a load.
"""
import json
import os
import sys
import time
import warnings

import numpy as np

from .graph import ColumnSchema, ColumnSelector, Node, Schema, Tags

FORMAT_VERSION = 1


class WorkflowSerializationError(Exception):
    """Raised when a workflow cannot be (de)serialized."""


# ------------------------------------------------------------------------------- small pieces
def _dtype_to_dict(dt):
    if dt is None:
        return None
    try:
        return {"name": str(np.dtype(dt))}
    except TypeError:
        return {"name": str(dt)}


def _dtype_from_dict(d):
    if not d:
        return None
    name = d["name"] if isinstance(d, dict) else d
    try:
        return np.dtype(name)
    except TypeError:
        return None


def _tags_to_list(tags):
    return [f"Tags.{t.name}" if isinstance(t, Tags) else str(t) for t in (tags or [])]


def _tags_from_list(items):
    out = []
    for s in items or []:
        name = str(s).split(".")[-1]
        try:
            out.append(Tags[name.upper()])
        except KeyError:
            pass                      # tags outside this engine's scope are dropped
    return out


def _json_safe(v):
    if isinstance(v, dict):
        return {str(k): _json_safe(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [_json_safe(x) for x in v]
    if isinstance(v, (np.integer,)):
        return int(v)
    if isinstance(v, (np.floating,)):
        return float(v)
    if isinstance(v, np.dtype) or isinstance(v, type):
        return str(np.dtype(v))
    return v


def _schema_to_list(schema):
    if schema is None:
        return None
    return [{"name": c.name, "tags": _tags_to_list(c.tags), "properties": _json_safe(c.properties),
             "dtype": _dtype_to_dict(c.dtype), "is_list": bool(c.is_list), "is_ragged": bool(c.is_ragged)}
            for c in schema]


def _schema_from_list(items):
    if items is None:
        return None
    return Schema([ColumnSchema(d["name"], _dtype_from_dict(d.get("dtype")), _tags_from_list(d.get("tags")),
                                d.get("properties") or {}, bool(d.get("is_list")), bool(d.get("is_ragged")))
                   for d in items])


def _selector_to_dict(sel):
    if sel is None:
        return None
    # "names" is what the reference stores; the grouping of multi-column groups is kept beside it
    return {"names": list(sel.names), "tags": [], "grouped_names": [list(g) if isinstance(g, tuple) else g
                                                                     for g in sel.grouped_names]}


def _selector_from_dict(d):
    if d is None:
        return None
    return ColumnSelector(d.get("grouped_names") or d["names"])


def _paths_to_records(paths: dict, artifact_dir):
    out = []
    for k, v in (paths or {}).items():
        out.append({"key": list(k) if isinstance(k, tuple) else [k], "path": os.path.relpath(str(v), artifact_dir)})
    return out


def _records_to_paths(records, artifact_dir):
    out = {}
    for r in records or []:
        k = tuple(r["key"]) if len(r["key"]) > 1 else r["key"][0]
        out[k] = os.path.join(artifact_dir, r["path"])
    return out


# ------------------------------------------------------------------------- operator registry
def _np_str(dt):
    return {"name": np.dtype(dt).str} if dt is not None else None


def _categorify_to(op, adir):
    cats = _paths_to_records(op.export_artifacts(adir), adir)      # the live op keeps its own paths
    params = {"freq_threshold": op.freq_threshold, "cat_cache": op.cat_cache if isinstance(op.cat_cache, str) else "host",
              "dtype": _np_str(op.dtype), "on_host": op.on_host, "encode_type": op.encode_type,
              "name_sep": op.name_sep, "search_sorted": op.search_sorted, "num_buckets": _json_safe(op.num_buckets),
              "max_size": _json_safe(op.max_size), "single_table": op.single_table,
              "cardinality_memory_limit": str(op.cardinality_memory_limit) if op.cardinality_memory_limit is not None
              else None, "split_out": _json_safe(op.split_out), "split_every": _json_safe(op.split_every)}
    return params, {"categories": cats, "storage_name": {str(k): str(v) for k, v in op.storage_name.items()}}


def _categorify_from(params, state, adir):
    from .ops.categorify import Categorify
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        op = Categorify(freq_threshold=params.get("freq_threshold", 0), cat_cache=params.get("cat_cache", "host"),
                        dtype=_dtype_from_dict(params.get("dtype")), on_host=params.get("on_host", True),
                        encode_type=params.get("encode_type", "joint"), name_sep=params.get("name_sep", "_"),
                        search_sorted=params.get("search_sorted", False), num_buckets=params.get("num_buckets"),
                        max_size=params.get("max_size", 0), single_table=params.get("single_table", False),
                        cardinality_memory_limit=params.get("cardinality_memory_limit"),
                        split_out=params.get("split_out", 1), split_every=params.get("split_every", 8))
    for k, v in _records_to_paths(state.get("categories"), adir).items():
        dict.__setitem__(op.categories, k, v)
    op.out_path = adir
    op.storage_name = dict(state.get("storage_name", {}))
    return op


def _moments_to(attr_a, attr_b):
    def f(op, adir):
        return ({"out_dtype": _dtype_to_dict(op.out_dtype)},
                {attr_a: {str(k): float(v) for k, v in getattr(op, attr_a).items()},
                 attr_b: {str(k): float(v) for k, v in getattr(op, attr_b).items()}})
    return f


def _moments_from(cls_name, attr_a, attr_b):
    def f(params, state, adir):
        from .ops import normalize
        op = getattr(normalize, cls_name)(out_dtype=_dtype_from_dict(params.get("out_dtype")))
        setattr(op, attr_a, {k: float(v) for k, v in state.get(attr_a, {}).items()})
        setattr(op, attr_b, {k: float(v) for k, v in state.get(attr_b, {}).items()})
        return op
    return f


def _join_groupby_to(op, adir):
    cats = _paths_to_records(op.export_tables(adir), adir)
    params = {"cont_cols": list(op._cont_names.names) if op._cont_names is not None else None, "stats": list(op.stats),
              "split_out": op.split_out, "split_every": op.split_every, "on_host": op.on_host,
              "cat_cache": op.cat_cache if isinstance(op.cat_cache, str) else "host", "name_sep": op.name_sep}
    return params, {"categories": cats, "storage_name": {str(k): str(v) for k, v in op.storage_name.items()}}


def _join_groupby_from(params, state, adir):
    from .ops.join_groupby import JoinGroupby
    op = JoinGroupby(cont_cols=params.get("cont_cols"), stats=tuple(params.get("stats", ("count",))),
                     split_out=params.get("split_out"), split_every=params.get("split_every"),
                     on_host=params.get("on_host", True), cat_cache=params.get("cat_cache", "host"),
                     name_sep=params.get("name_sep", "_"))
    op.categories = _records_to_paths(state.get("categories"), adir)
    op.out_path = adir
    op.storage_name = dict(state.get("storage_name", {}))
    return op


def _target_encoding_to(op, adir):
    stats = _paths_to_records(op.export_tables(adir), adir)
    params = {"target_cols": list(op.target_columns), "target_mean": _json_safe(op.target_mean), "kfold": op.kfold,
              "fold_seed": op.fold_seed, "p_smooth": op.p_smooth, "out_col": op.out_col,
              "out_dtype": _np_str(op.out_dtype), "name_sep": op.name_sep, "drop_folds": op.drop_folds}
    return params, {"stats": stats, "means": {str(k): float(v) for k, v in op.means.items()}}


def _target_encoding_from(params, state, adir):
    from .ops.target_encoding import TargetEncoding
    op = TargetEncoding(target=params.get("target_cols", []), target_mean=params.get("target_mean"),
                        kfold=params.get("kfold", 3), fold_seed=params.get("fold_seed", 42),
                        p_smooth=params.get("p_smooth", 20), out_col=params.get("out_col"),
                        out_dtype=_dtype_from_dict(params.get("out_dtype")), name_sep=params.get("name_sep", "_"),
                        drop_folds=params.get("drop_folds", True))
    op.stats = _records_to_paths(state.get("stats"), adir)
    op.means = {k: float(v) for k, v in state.get("means", {}).items()}
    op.out_path = adir
    return op


def _registry():
    from . import ops
    return {
        "nvtabular.ops.categorify.Categorify": (ops.Categorify, _categorify_to, _categorify_from),
        "nvtabular.ops.normalize.Normalize": (ops.Normalize, _moments_to("means", "stds"),
                                              _moments_from("Normalize", "means", "stds")),
        "nvtabular.ops.normalize.NormalizeMinMax": (ops.NormalizeMinMax, _moments_to("mins", "maxs"),
                                                    _moments_from("NormalizeMinMax", "mins", "maxs")),
        "nvtabular.ops.fill.FillMissing": (
            ops.FillMissing, lambda op, adir: ({"fill_val": op.fill_val, "add_binary_cols": op.add_binary_cols}, {}),
            lambda p, s, adir: ops.FillMissing(fill_val=p.get("fill_val", 0), add_binary_cols=p.get("add_binary_cols", False))),
        "nvtabular.ops.clip.Clip": (
            ops.Clip, lambda op, adir: ({"min_value": op.min_value, "max_value": op.max_value}, {}),
            lambda p, s, adir: ops.Clip(min_value=p.get("min_value"), max_value=p.get("max_value"))),
        "nvtabular.ops.logop.LogOp": (ops.LogOp, lambda op, adir: ({}, {}), lambda p, s, adir: ops.LogOp()),
        "nvtabular.ops.hash_bucket.HashBucket": (
            ops.HashBucket, lambda op, adir: ({"num_buckets": _json_safe(op.num_buckets)}, {}),
            lambda p, s, adir: ops.HashBucket(num_buckets=p["num_buckets"])),
        "nvtabular.ops.join_groupby.JoinGroupby": (ops.JoinGroupby, _join_groupby_to, _join_groupby_from),
        "nvtabular.ops.target_encoding.TargetEncoding": (ops.TargetEncoding, _target_encoding_to, _target_encoding_from),
        # graph_serializer.py:450-471 of the reference
        "nvtabular.ops.list_slice.ListSlice": (
            ops.ListSlice, lambda op, adir: ({"start": op.start, "end": op.end, "pad": op.pad, "pad_value": op.pad_value}, {}),
            lambda p, s, adir: ops.ListSlice(start=p["start"], end=p.get("end"), pad=p.get("pad", False),
                                             pad_value=p.get("pad_value", 0.0))),
    }


# operators the reference's serializer refuses (graph_serializer.py:919-929); refusing them too keeps
# graph.json readable by either implementation
_DEFERRED = {"Groupby"}


_KIND_CLASS = {"input": "merlin.dag.ops.selection.SelectionOp", "concat": "merlin.dag.ops.concat_columns.ConcatColumns",
               "subtract": "merlin.dag.ops.subtraction.SubtractionOp", "subset": "merlin.dag.ops.subset_columns.SubsetColumns"}
_CLASS_KIND = {v: k for k, v in _KIND_CLASS.items()}


# ----------------------------------------------------------------------------------- public
def save_workflow(workflow, path):
    """Workflow.save (reference workflow.py:256-296): metadata.json + graph.json + artifacts/."""
    import pandas as pd
    from . import __version__ as version
    path = str(path)
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "metadata.json"), "w") as f:
        json.dump({"versions": {"nvtabular": version, "pandas": pd.__version__, "python": sys.version},
                   "generated_timestamp": int(time.time())}, f)
    reg = _registry()
    by_cls = {cls: (name, to) for name, (cls, to, _) in reg.items()}
    nodes = workflow.output_node.topo_order()
    ids = {id(n): i for i, n in enumerate(nodes)}
    records = []
    for n in nodes:
        i = ids[id(n)]
        adir = os.path.join(path, "artifacts", f"node_{i}")
        if n.kind == "op":
            if type(n.op).__name__ in _DEFERRED:
                raise NotImplementedError(
                    f"The operator '{type(n.op).__name__}' is not yet supported by the JSON workflow "
                    "serializer. Please open an issue or use a supported operator.")
            entry = by_cls.get(type(n.op))
            if entry is None:
                raise WorkflowSerializationError(f"no serializer for operator {type(n.op).__name__}")
            op_class, to = entry
            params, state = to(n.op, adir)
        else:
            op_class = _KIND_CLASS[n.kind]
            params, state = ({"selector": _selector_to_dict(n.selector)} if n.selector is not None else {}), {}
        records.append({"id": i, "op_class": op_class, "op_params": _json_safe(params), "op_state": _json_safe(state),
                        "parent_ids": [ids[id(p)] for p in n.parents],
                        "dependency_ids": [ids[id(d)] for d in n.dependencies],
                        "selector": _selector_to_dict(n.selector),
                        "input_schema": _schema_to_list(n.input_schema),
                        "output_schema": _schema_to_list(n.output_schema)})
    graph = {"format_version": FORMAT_VERSION, "output_node_id": ids[id(workflow.output_node)], "nodes": records,
             "input_schema": _schema_to_list(workflow.input_schema),
             "output_schema": _schema_to_list(workflow._output_schema)}
    with open(os.path.join(path, "graph.json"), "w") as f:
        json.dump(graph, f, indent=2)


def load_workflow(path, client=None):
    """Workflow.load (reference workflow.py:298-348)."""
    from . import __version__ as version
    from .workflow import Workflow
    path = str(path)
    with open(os.path.join(path, "metadata.json")) as f:
        meta = json.load(f)
    stored = meta.get("versions", {}).get("nvtabular")
    if stored is not None and stored.split(".")[:2] != version.split(".")[:2]:
        warnings.warn(f"Loading workflow generated with nvtabular version {stored} - but we are running "
                      f"nvtabular {version}. This might cause issues")
    with open(os.path.join(path, "graph.json")) as f:
        graph = json.load(f)
    if graph.get("format_version", 1) != FORMAT_VERSION:
        raise WorkflowSerializationError(f"Unsupported graph.json format_version={graph.get('format_version')}")
    reg = _registry()
    node_map = {}
    for r in sorted(graph["nodes"], key=lambda r: r["id"]):
        adir = os.path.join(path, "artifacts", f"node_{r['id']}")
        cls = r.get("op_class")
        node = Node()
        sel = _selector_from_dict(r.get("selector"))
        if cls in _CLASS_KIND:
            node.kind = _CLASS_KIND[cls]
            node.selector = sel if sel is not None else _selector_from_dict((r.get("op_params") or {}).get("selector"))
        else:
            entry = reg.get(cls)
            if entry is None:
                raise WorkflowSerializationError(f"Unknown operator class '{cls}' in graph.json.")
            node.kind = "op"
            node.op = entry[2](r.get("op_params") or {}, r.get("op_state") or {}, adir)
            node.selector = None
        node.input_schema = _schema_from_list(r.get("input_schema"))
        node.output_schema = _schema_from_list(r.get("output_schema"))
        for pid in r.get("parent_ids", []):
            node.add_parent(node_map[pid])
        for did in r.get("dependency_ids", []):
            node.dependencies.append(node_map[did])
            node_map[did].children.append(node)
        node_map[r["id"]] = node
    wf = Workflow(node_map[graph["output_node_id"]], client=client)
    wf.input_schema = _schema_from_list(graph.get("input_schema"))
    wf._output_schema = _schema_from_list(graph.get("output_schema"))
    return wf
