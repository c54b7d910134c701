"""Groupby (reference nvtabular/ops/groupby.py): per-partition sort + group-by + aggregation for
session-based pipelines.  Each partition is ordered once on the device by (group keys, sort
columns) with nvtb_sort_rows, cut into groups once (nvtb_segments), and every output column is
one more kernel over that order (csrc/groupby.cu).  Like the reference, rows never move between
partitions: shuffle the Dataset by the group keys first (Dataset.shuffle_by_keys)."""
from typing import Dict, List, Tuple

import numpy as np

from .. import engine
from ..column import Column, DeviceFrame
from ..graph import ColumnSchema, ColumnSelector, Schema
from .base import Operator

_SCALAR_AGGS = ("count", "sum", "mean", "min", "max", "std", "var", "first", "last")
_SORTED_AGGS = ("median", "nunique")
_NUMERIC_ONLY = ("sum", "mean", "std", "var", "median")
_KNOWN = set(_SCALAR_AGGS) | set(_SORTED_AGGS) | {"list"}
# reference _compute_dtype, groupby.py:190-203
_AGG_DTYPES = {"count": np.dtype("int32"), "nunique": np.dtype("int32"), "mean": np.dtype("float32"),
               "var": np.dtype("float32"), "std": np.dtype("float32"), "median": np.dtype("float32"),
               "sum": np.dtype("float32")}


def _is_object(dtype) -> bool:
    try:
        return dtype is not None and np.dtype(dtype) == np.dtype("O")
    except TypeError:
        return False


def _as_list(v):
    return list(v) if isinstance(v, (list, tuple)) else [v]


class Groupby(Operator):
    """Groupby Transformation (reference groupby.py:26-112).

    groupby_cols : str or list of str, the group keys (rows with a null key are dropped)
    sort_cols    : str or list of str, a stable sort applied before grouping (nulls last)
    aggs         : str, list or dict {column | "__all__": agg or [aggs]} over count, sum, mean, min,
                   max, std, var, median, nunique, list, first, last (`list` itself means "list")
    name_sep     : separator of the output names `<column><name_sep><agg>`
    ascending    : direction of sort_cols; first / last swap when False (groupby.py:290-297)
    """

    def __init__(self, groupby_cols=None, sort_cols=None, aggs="list", name_sep="_", ascending=True):
        super().__init__()
        self.groupby_cols = [groupby_cols] if isinstance(groupby_cols, str) else list(groupby_cols or [])
        self.sort_cols = [sort_cols] if isinstance(sort_cols, str) else list(sort_cols or [])
        self.ascending = ascending
        if isinstance(aggs, str) or aggs is list:
            aggs = {"__all__": [aggs]}
        elif isinstance(aggs, (list, tuple)):
            aggs = {"__all__": list(aggs)}
        self.aggs: Dict[str, List[str]] = {}
        for col, v in aggs.items():
            names = []
            for a in _as_list(v):
                a = "list" if a is list else a
                if a not in _KNOWN:
                    raise ValueError(f"Groupby: unsupported aggregation {a!r} for column {col!r}")
                if a not in names:
                    names.append(a)
            self.aggs[col] = names
        self.name_sep = name_sep

    @property
    def dependencies(self):
        return self.groupby_cols

    # ---------------------------------------------------------------------------- naming
    def _plan(self, col_selector: ColumnSelector) -> List[Tuple[str, str, str]]:
        """[(output name, source column, agg)]: keys in the selector first (agg None), then the
        columns and aggs in the order given (reference _get_agg_dicts, groupby.py:263-279, which
        maps "__all__" to every selected non-key column)"""
        names = col_selector.names
        plan = [(k, k, None) for k in self.groupby_cols if k in names]
        allowed = [c for c in names if c not in self.groupby_cols]
        if "__all__" in self.aggs:
            per_col = [(c, self.aggs["__all__"]) for c in allowed]
        else:
            per_col = [(c, a) for c, a in self.aggs.items() if c in allowed]
        for col, aggs in per_col:
            for a in aggs:
                plan.append((f"{col}{self.name_sep}{a}", col, a))
        return plan

    def column_mapping(self, col_selector):
        return {out: [src] for out, src, _ in self._plan(col_selector)}

    def compute_output_schema(self, input_schema: Schema, col_selector: ColumnSelector) -> Schema:
        out = []
        for name, src, agg in self._plan(col_selector):
            s = input_schema[src] if src in input_schema else ColumnSchema(src)
            self._check(src, agg, s.is_list, _is_object(s.dtype))
            cs = ColumnSchema(name, s.dtype, s.tags, s.properties, s.is_list, s.is_ragged)
            if agg == "list":
                cs = cs.with_dtype(s.dtype, True, True)
            elif agg in _AGG_DTYPES:
                cs = cs.with_dtype(_AGG_DTYPES[agg], False, False)
            elif agg in ("min", "max"):
                cs = cs.with_dtype(s.dtype, False, False)
            out.append(cs)
        return Schema(out)

    @staticmethod
    def _check(col, agg, is_list, is_string):
        if agg is None:
            return
        if is_list and agg not in ("first", "last"):
            what = "nested lists are not supported" if agg == "list" else "only first / last apply to list columns"
            raise ValueError(f"Groupby: {agg!r} of list column {col!r}: {what}")
        if is_string and agg in _NUMERIC_ONLY:
            raise TypeError(f"Groupby: {agg!r} of string column {col!r} is not defined")

    # ------------------------------------------------------------------------- transform
    def transform(self, col_selector: ColumnSelector, df: DeviceFrame) -> DeviceFrame:
        plan = self._plan(col_selector)
        keys = [self._get(df, k) for k in self.groupby_cols]
        if not keys:
            raise ValueError("Groupby needs groupby_cols")
        for k, c in zip(self.groupby_cols, keys):
            if c.is_list:
                raise ValueError(f"Groupby: key column {k!r} is a list column")
        sorts = [self._get(df, s) for s in self.sort_cols]
        desc = [False] * len(keys) + [not self.ascending] * len(sorts)
        perm, n_kept = engine.sort_rows(keys + sorts, desc, n_drop_null=len(keys))
        offsets, n_groups, n_rows = engine.segments(keys, perm, n_kept)
        starts, ends = offsets[:-1], offsets[1:]

        by_col: Dict[str, List[str]] = {}
        for _, src, agg in plan:
            if agg is not None:
                by_col.setdefault(src, []).append(agg)
        results: Dict[Tuple[str, str], Column] = {}
        for src, aggs in by_col.items():
            col = self._get(df, src)
            for a in aggs:
                self._check(src, a, col.is_list, col.is_string)
            # first / last are element 0 / -1 of the sorted list, swapped when descending
            swap = {"first": "last", "last": "first"} if not self.ascending else {}
            if col.is_list:
                for a in aggs:
                    eff = swap.get(a, a)
                    idx, shift = (starts, 0) if eff == "first" else (ends, -1)
                    results[(src, a)] = engine.list_slice(col, 0, np.iinfo(np.int64).max, perm=perm, idx=idx,
                                                          shift=shift, n_rows=n_groups)
                continue
            scalar = [swap.get(a, a) for a in aggs if a in _SCALAR_AGGS]
            if scalar:
                got = engine.segment_agg(col, perm, offsets, n_groups, list(dict.fromkeys(scalar)))
                for a in aggs:
                    if a in _SCALAR_AGGS:
                        results[(src, a)] = got[swap.get(a, a)]
            if any(a in _SORTED_AGGS for a in aggs):
                vperm, _ = engine.sort_rows(keys + [col], [False] * (len(keys) + 1), n_drop_null=len(keys))
                got = engine.segment_sorted_agg(col, vperm, offsets, n_groups, n_rows,
                                                median="median" in aggs, nunique="nunique" in aggs)
                for a in _SORTED_AGGS:
                    if a in got:
                        results[(src, a)] = got[a]
            if "list" in aggs:
                leaves = engine.gather_rows(col, perm, n_rows)
                leaves.offsets = offsets
                results[(src, "list")] = leaves

        out = DeviceFrame()
        for name, src, agg in plan:
            if agg is None:
                out[name] = engine.gather_rows(self._get(df, src), perm, n_groups, idx=starts)
            else:
                out[name] = results[(src, agg)]
        return out
