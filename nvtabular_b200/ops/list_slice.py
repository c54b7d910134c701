"""ListSlice (reference nvtabular/ops/list_slice.py): Python slicing of every row of a list
column, optionally padded at the end to a fixed length.  Two kernels replace the reference's
numba _calculate_row_sizes / _slice_rows (list_slice.py:180-228): per-row sizes + scan, then a
load-balanced element copy (csrc/groupby.cu nvtb_list_slice_offsets / nvtb_list_slice)."""
import numpy as np

from .. import engine
from ..column import DeviceFrame
from ..graph import ColumnSelector, Tags
from .base import Operator

_UNBOUNDED = np.iinfo(np.int64).max


class ListSlice(Operator):
    """Slices a list column (reference list_slice.py:28-75).

    start     : the start of the slice, or its end when `end` is not given and start > 0
    end       : the end of the slice (negative counts from the row end)
    pad       : pad every row at the end to `max_elements` values
    pad_value : the padding value, cast to the list's dtype
    """

    def __init__(self, start, end=None, pad=False, pad_value=0.0):
        super().__init__()
        self.start = start
        self.end = end
        self.pad = pad
        self.pad_value = pad_value
        # constructor normalisation of list_slice.py:58-75
        if self.start > 0 and self.end is None:
            self.end = self.start
            self.start = 0
        if self.end is None:
            self.end = _UNBOUNDED
        if self.start < 0:
            self.max_elements = -(self.start if self.end > 0 else self.start - self.end)
        else:
            self.max_elements = self.end - self.start
        if self.pad and not 0 <= self.max_elements < _UNBOUNDED:
            raise ValueError(f"ListSlice(pad=True) needs a slice of bounded, non-negative length; "
                             f"ListSlice({start}, {end}) has {self.max_elements}")

    def transform(self, col_selector: ColumnSelector, df: DeviceFrame) -> DeviceFrame:
        out = DeviceFrame()
        for name in col_selector.names:
            col = self._get(df, name)
            if not col.is_list:
                raise TypeError(f"ListSlice: column {name!r} is not a list column")
            out[name] = engine.list_slice(col, self.start, self.end, self.pad, self.max_elements, self.pad_value)
        return out

    @property
    def output_tags(self):
        return [Tags.LIST]

    def _compute_dtype(self, col_schema, input_schema):
        cs = super()._compute_dtype(col_schema, input_schema)
        return cs.with_dtype(cs.dtype, True, not self.pad)

    def _compute_properties(self, col_schema, input_schema):
        cs = super()._compute_properties(col_schema, input_schema)
        value_count = {"min": 0, "max": None}                 # list_slice.py:150-160
        if self.max_elements != _UNBOUNDED:
            value_count["max"] = self.max_elements
            if self.pad:
                value_count["min"] = self.max_elements
        return cs.with_properties({"value_count": value_count})
