"""CPU oracle of the session ops — TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

pandas restatements of reference nvtabular/ops/groupby.py (Groupby.__init__ :76-112, transform
:114-150, _apply_aggs :213-240, _get_agg_dicts / _ensure_agg_dict :243-259, _first_or_last
:290-319, _compute_dtype :190-203) and of the CPU branch of ListSlice.transform
(nvtabular/ops/list_slice.py:58-75, 89-103).

A fourth documented deviation, after the three of oracle/__init__.py:
  4. the sort by sort_cols uses kind="stable" (groupby.py:116 calls sort_values with pandas'
     default quicksort on one column, which leaves the order of ties unspecified).
Rows are handled as Python lists by ListSlice's CPU branch, which is the branch that pads (the
ndarray branch of list_slice.py:95-99 drops the padding it computes)."""
import numpy as np
import pandas as pd

INT64_MAX = np.iinfo(np.int64).max
_AGG_DTYPES = {"count": "int32", "nunique": "int32", "mean": "float32", "median": "float32",
               "std": "float32", "var": "float32", "sum": "float32"}


def normalize_aggs(aggs):
    """Groupby.__init__ (groupby.py:92-108): str / list / dict -> {column | "__all__": [aggs]}"""
    if isinstance(aggs, str) or aggs is list:
        aggs = {"__all__": [aggs]}
    elif isinstance(aggs, (list, tuple)):
        aggs = {"__all__": list(aggs)}
    out = {}
    for col, v in aggs.items():
        vals = v if isinstance(v, (list, tuple)) else [v]
        out[col] = list(dict.fromkeys("list" if a is list else a for a in vals))
    return out


def groupby(df: pd.DataFrame, groupby_cols, sort_cols=None, aggs="list", name_sep="_", ascending=True,
            columns=None) -> pd.DataFrame:
    """Groupby.transform on one partition.  `columns` is the op's selector (default: every column)."""
    groupby_cols = [groupby_cols] if isinstance(groupby_cols, str) else list(groupby_cols)
    sort_cols = [sort_cols] if isinstance(sort_cols, str) else list(sort_cols or [])
    columns = list(df.columns) if columns is None else list(columns)
    aggs = normalize_aggs(aggs)
    if sort_cols:                                                         # groupby.py:116 (+ deviation 4)
        df = df.sort_values(sort_cols, ascending=ascending, kind="stable", na_position="last",
                            ignore_index=True)
    allowed = [c for c in columns if c not in groupby_cols]               # _get_agg_dicts
    if "__all__" in aggs:
        per_col = [(c, aggs["__all__"]) for c in allowed]
    else:
        per_col = [(c, a) for c, a in aggs.items() if c in allowed]
    g = df.groupby(groupby_cols, sort=True, dropna=True)
    out = {}
    keys = g.size().reset_index()[groupby_cols]
    for k in groupby_cols:
        if k in columns:
            out[k] = keys[k].to_numpy()
    for col, col_aggs in per_col:
        lists = g[col].agg(list) if any(a in ("list", "first", "last") for a in col_aggs) else None
        for a in col_aggs:
            name = f"{col}{name_sep}{a}"
            if a == "list":
                vals = lists.to_numpy()
            elif a in ("first", "last"):                                  # _first_or_last
                take_first = (a == "first") == bool(ascending)
                picked = [r[0] if take_first else r[-1] for r in lists]
                nested = bool(picked) and isinstance(picked[0], (list, np.ndarray))
                vals = pd.Series(picked, dtype=object if nested else None).to_numpy()
            elif a in _AGG_DTYPES:                                        # _apply_aggs casts, :232-238
                vals = getattr(g[col], a)().to_numpy(dtype="float64", na_value=np.nan).astype(_AGG_DTYPES[a])
            else:
                vals = getattr(g[col], a)().to_numpy()
            out[name] = vals
    return pd.DataFrame({k: pd.Series(list(v), dtype=object) if v.dtype == object else pd.Series(v)
                         for k, v in out.items()})


def list_slice_bounds(start, end=None):
    """ListSlice.__init__ (list_slice.py:64-75) -> (start, end, max_elements)"""
    if start > 0 and end is None:
        end, start = start, 0
    if end is None:
        end = INT64_MAX
    if start < 0:
        max_elements = -(start if end > 0 else start - end)
    else:
        max_elements = end - start
    return start, end, max_elements


def list_slice(rows, start, end=None, pad=False, pad_value=0.0):
    """the CPU branch of ListSlice.transform (list_slice.py:89-103) on a sequence of rows"""
    start, end, max_elements = list_slice_bounds(start, end)
    out = []
    for row in rows:
        v = list(row)[start:end]
        if pad and len(v) < max_elements:
            v.extend([pad_value] * (max_elements - len(v)))
        out.append(v)
    return out
