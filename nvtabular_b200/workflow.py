"""Workflow.fit / transform / fit_transform (reference
nvtabular/workflow/workflow.py:45-358).  The reference delegates to
merlin.dag's DaskExecutor / LocalExecutor (workflow.py:74,209,242,254); here the
operator DAG is executed directly on device-resident partitions:

  fit        StatOperator nodes are fitted in dependency "phases" exactly like
             DaskExecutor.fit: a node is ready once every StatOperator upstream
             of it has been fitted; its input is the dataset pushed through
             those upstream nodes.
  transform  every partition is pushed through the DAG in topological order;
             `Dataset` inputs are transformed lazily (on `.compute()` /
             `.to_ddf()` / iteration), DataFrame inputs eagerly.
"""
import json
import os
from typing import Dict, List, Optional

import pandas as pd

from .column import DeviceFrame
from .dataset import Dataset
from .graph import ColumnSchema, ColumnSelector, Node, Schema
from .ops.base import Operator, StatOperator
from .ops.fill import materialize_many


def _merge_frames(node: Node, sources: List[Node], frames: List[DeviceFrame]) -> DeviceFrame:
    """the columns of several upstream frames as one frame; they must have the same rows (a
    Groupby upstream of only some of them changes the row count)"""
    lens = {id(s): len(f) for s, f in zip(sources, frames) if f.columns}
    if len(set(lens.values())) > 1:
        detail = ", ".join(f"{s!r}: {lens[id(s)]} rows" for s in sources if id(s) in lens)
        raise ValueError(f"{node!r} merges inputs with different row counts ({detail})")
    out = DeviceFrame()
    for f in frames:
        for k, v in f.items():
            out[k] = v
    return out


def _execute_node(node: Node, root: DeviceFrame, cache: Dict[int, DeviceFrame]) -> DeviceFrame:
    hit = cache.get(id(node))
    if hit is not None:
        return hit
    if node.kind == "input":
        missing = [n for n in node.selector.names if n not in root]
        if missing:
            raise ValueError(f"Missing columns {missing} found in operator input")
        out = root[node.selector.names]
    else:
        frames = [_execute_node(p, root, cache) for p in node.upstream]
        if node.kind in ("concat",):
            out = _merge_frames(node, node.upstream, frames)
        elif node.kind == "subtract":
            out = frames[0].drop(node.selector.names)
        elif node.kind == "subset":
            out = frames[0][node.selector.names]
        else:
            inp = _merge_frames(node, node.upstream, frames)
            if not node.op.fuses_fill:
                names = inp.columns
                cols = materialize_many([inp[n] for n in names])
                inp = DeviceFrame(dict(zip(names, cols)))
            with _nvtx(f"{type(node.op).__name__}_op"):
                res = node.op.transform(node.input_columns, inp)
            keep = node.output_columns.names
            out = DeviceFrame({k: res[k] for k in keep if k in res})
    cache[id(node)] = out
    return out


class _nvtx:
    """NVTX range per operator and phase — the reference's @annotate("<Op>_op" / "<Op>_fit",
    domain="nvt_python") ranges (nvtabular/ops/categorify.py:345,477; ops/clip.py:45), visible in
    Nsight Systems timelines.  NVTB_NVTX=0 turns them off."""
    _on = None

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _nvtx._on is None:
            import torch
            _nvtx._on = torch.cuda.is_available() and os.environ.get("NVTB_NVTX", "1") != "0"
        if _nvtx._on:
            import torch
            torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        if _nvtx._on:
            import torch
            torch.cuda.nvtx.range_pop()
        return False


def _finalize_frame(frame: DeviceFrame) -> DeviceFrame:
    names = frame.columns
    return DeviceFrame(dict(zip(names, materialize_many([frame[n] for n in names]))))


class _UpstreamPartitions:
    """The `ddf` handed to StatOperator.fit: the dataset's partitions pushed through
    the parents (and dependencies) of one node."""

    def __init__(self, dataset: Dataset, node: Node):
        self.dataset = dataset
        self.node = node

    def __iter__(self):
        for part in self.dataset.partitions():
            cache: Dict[int, DeviceFrame] = {}
            ups = self.node.upstream
            yield _merge_frames(self.node, ups, [_execute_node(up, part, cache) for up in ups])


class Workflow:
    def __init__(self, output_node, client=None):
        self.output_node = Node.construct_from(output_node)
        self.client = client           # accepted; there is no dask
        self.input_schema: Optional[Schema] = None
        self._output_schema: Optional[Schema] = None

    # ------------------------------------------------------------------------ fit
    def fit(self, dataset: Dataset) -> "Workflow":
        self.clear_stats()
        order = self.output_node.topo_order()
        stat_nodes = [n for n in order if n.kind == "op" and isinstance(n.op, StatOperator)]
        fitted = set()

        def upstream_stats(n):
            return [u for u in n.topo_order() if u is not n and u.kind == "op" and isinstance(u.op, StatOperator)]

        while stat_nodes:
            ready = [n for n in stat_nodes if all(id(u) in fitted for u in upstream_stats(n))]
            if not ready:
                raise RuntimeError("failed to find dependency-free StatOperator to fit")
            # ops of one phase are independent: fit the ones whose fit ends in a blocking
            # device->host read (Normalize's moments) FIRST, so that the read waits on an
            # almost empty stream instead of draining everything Categorify has queued
            ready.sort(key=lambda n: 0 if getattr(n.op, "fit_blocks_host", False) else 1)
            for n in ready:
                with _nvtx(f"{type(n.op).__name__}_fit"):
                    stats = n.op.fit(n.input_columns, _UpstreamPartitions(dataset, n))
                with _nvtx(f"{type(n.op).__name__}_fit_finalize"):
                    n.op.fit_finalize(stats)
                fitted.add(id(n))
            stat_nodes = [n for n in stat_nodes if id(n) not in fitted]
        self.fit_schema(dataset.schema)
        return self

    def fit_schema(self, input_schema: Schema) -> "Workflow":
        schemas: Dict[int, Schema] = {}
        for n in self.output_node.topo_order():
            if n.kind == "input":
                s = Schema([input_schema[c] if c in input_schema else ColumnSchema(c) for c in n.selector.names])
            else:
                merged = Schema()
                for u in n.upstream:
                    merged = merged + schemas[id(u)]
                if n.kind == "concat":
                    s = merged
                elif n.kind == "subtract":
                    s = merged.without(n.selector.names)
                elif n.kind == "subset":
                    s = merged.select_by_name(n.selector.names)
                else:
                    n.input_schema = merged
                    s = n.op.compute_output_schema(merged, n.input_columns)
            n.output_schema = s
            schemas[id(n)] = s
        roots = self.output_node.root_columns()
        self.input_schema = Schema([input_schema[c] if c in input_schema else ColumnSchema(c) for c in roots])
        self._output_schema = schemas[id(self.output_node)]
        return self

    # ------------------------------------------------------------------ transform
    def _transform_frame(self, frame: DeviceFrame) -> DeviceFrame:
        return _finalize_frame(_execute_node(self.output_node, frame, {}))

    def transform(self, data):
        if isinstance(data, Dataset):
            return Dataset(data, _transform=self._transform_frame, base_dataset=data._base_dataset if data._base_dataset is not None else data,
                           schema=self._output_schema)
        if isinstance(data, pd.DataFrame):
            if self._output_schema is None:
                raise ValueError("no output schema")
            return self._transform_frame(DeviceFrame.from_pandas(data.reset_index(drop=True))).to_pandas()
        if isinstance(data, DeviceFrame):
            return self._transform_frame(data)
        raise NotImplementedError(
            f"Workflow.transform received an unsupported type: {type(data)} "
            "Supported types are a `merlin.io.Dataset` or DataFrame (pandas or cudf)")

    def fit_transform(self, dataset: Dataset) -> Dataset:
        self.fit(dataset)
        return self.transform(dataset)

    # ----------------------------------------------------------------------- misc
    def clear_stats(self):
        for n in self.output_node.topo_order():
            if n.kind == "op" and isinstance(n.op, StatOperator):
                n.op.clear()

    @property
    def output_schema(self) -> Optional[Schema]:
        return self._output_schema

    @property
    def input_dtypes(self):
        return {c.name: c.dtype for c in self.input_schema} if self.input_schema else None

    @property
    def output_dtypes(self):
        return {c.name: c.dtype for c in self._output_schema} if self._output_schema else None

    def get_subworkflow(self, subgraph_name):
        raise NotImplementedError("subgraphs are outside the hot-path scope (SURVEY.md §8)")

    def remove_inputs(self, input_cols) -> "Workflow":
        for n in self.output_node.topo_order():
            if n.kind == "input":
                n.selector = ColumnSelector([c for c in n.selector.names if c not in set(input_cols)])
        return self

    # save / load in the reference's layout: metadata.json + graph.json + artifacts/node_<id>/
    # (reference nvtabular/workflow/workflow.py:256-348, graph_serializer.py:1077-1165)
    def save(self, path):
        from .serialize import save_workflow
        save_workflow(self, path)

    @classmethod
    def load(cls, path, client=None) -> "Workflow":
        from .serialize import load_workflow
        return load_workflow(path, client)
