"""Dataset: the partitioned, device-resident table a Workflow runs on.

Stands in for merlin.io.Dataset (un-vendored; call sites reference
nvtabular/workflow/workflow.py:195-248, bench/examples/
dask-nvtabular-criteo-benchmark.py:216).  A partition is a DeviceFrame in HBM;
there is no dask graph — `to_ddf().compute()` simply brings a (lazily
transformed) dataset back as a pandas frame, as the reference's tests do.
"""
import os
from typing import Callable, Iterable, List, Optional, Union

import numpy as np
import pandas as pd
import torch

from .column import Column, DeviceFrame
from .graph import ColumnSchema, Schema


_COPY_STREAMS = {}


def _copy_stream(dev, which=0):
    key = (dev.index, which)
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _COPY_STREAMS[key]


def _schema_of(frame: DeviceFrame) -> Schema:
    cols = []
    for name, c in frame.items():
        cols.append(ColumnSchema(name, dtype=c.np_dtype, is_list=c.is_list, is_ragged=c.is_list))
    return Schema(cols)


class _Lazy:
    """What `Dataset.to_ddf()` returns: `.compute()` -> pandas DataFrame."""

    def __init__(self, ds: "Dataset", columns=None):
        self._ds = ds
        self._columns = columns

    def compute(self, scheduler=None, **kwargs) -> pd.DataFrame:
        frames = []
        for part in self._ds.partitions():
            if self._columns is not None:
                part = part[list(self._columns)]
            frames.append(part.to_pandas())
        if not frames:
            return pd.DataFrame()
        return pd.concat(frames, ignore_index=True) if len(frames) > 1 else frames[0]

    @property
    def npartitions(self):
        return self._ds.npartitions

    @property
    def columns(self):
        return self._ds.schema.column_names

    def head(self, n=5):
        return self.compute().head(n)

    def __getitem__(self, cols):
        return _Lazy(self._ds, [cols] if isinstance(cols, str) else list(cols))


class Dataset:
    """`Dataset(df)`, `Dataset([df0, df1])`, `Dataset(DeviceFrame)`, `Dataset(dict of tensors)`,
    `Dataset("file.parquet" | [paths])`.  `npartitions` splits a single host frame by rows
    (what `dd.from_pandas(df, npartitions=k)` does in the reference's tests)."""

    def __init__(self, data, engine=None, npartitions: Optional[int] = None, cpu: bool = False,
                 part_size=None, schema: Optional[Schema] = None, device=None,
                 _transform: Optional[Callable] = None, base_dataset=None, **kwargs):
        self._device = device
        # part_size: rows per partition for file sources (int), or None = one per row group;
        # byte strings ("1GB") are accepted like the reference and mapped through a nominal
        # 160 B/row (the Criteo-shaped row of SURVEY.md 8d)
        self._part_rows = None
        if part_size is not None:
            if isinstance(part_size, str):
                from .ops.categorify import _parse_bytes
                self._part_rows = max(64, int(_parse_bytes(part_size) // 160) // 64 * 64)
            else:
                self._part_rows = max(1, int(part_size))
        self.cache_on_device = kwargs.pop("cache_on_device", True)
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._transform = _transform
        # NOT `base_dataset or self`: a self-reference makes every Dataset a reference cycle, and the
        # HBM copies of its partitions then live until the cyclic GC happens to run (measured: 22 GB
        # per end-to-end step, allocator retries and second-long stalls in the following fits)
        self._base_dataset = base_dataset
        self.cpu = cpu     # accepted for API compatibility; there is no CPU engine
        self._parts: Optional[List[DeviceFrame]] = None
        self._source = data
        self._npartitions = npartitions
        if isinstance(data, Dataset):
            # same source, same partitioning: a Dataset that has not been ingested yet must split
            # the way its parent would (TargetEncoding draws its folds per partition)
            if data._parts is None:
                data._parts = data._ingest()
            self._source = data._source
            self._parts = data._parts
            self._npartitions = data._npartitions
            self._part_rows = data._part_rows
            self._device = data._device
            # a lazily transformed Dataset handed to another Workflow: CHAIN the transforms
            # (wf2.transform(wf1.transform(ds)) runs wf2 on wf1's output, like the reference)
            prev = data._transform
            if prev is not None and _transform is not None:
                self._transform = lambda part, _f=prev, _g=_transform: _g(_f(part))
            else:
                self._transform = _transform or prev
        self._schema = schema

    @property
    def base_dataset(self):
        return self._base_dataset if self._base_dataset is not None else self

    # --------------------------------------------------------------- ingestion
    def _ingest(self) -> List[DeviceFrame]:
        src = self._source
        if isinstance(src, (str, bytes)) or (isinstance(src, (list, tuple)) and src
                                             and all(isinstance(s, str) for s in src)):
            paths = [src] if isinstance(src, (str, bytes)) else list(src)
            paths = [os.fsdecode(p) for p in paths]
            expanded = []
            for p in paths:                     # a directory of part files, like merlin.io.Dataset
                if os.path.isdir(p):
                    expanded += sorted(os.path.join(p, f) for f in os.listdir(p)
                                       if f.endswith(".parquet") or f.endswith(".csv"))
                else:
                    expanded.append(p)
            if all(not p.endswith(".csv") for p in expanded):
                return self._ingest_parquet(expanded)
            host = [pd.read_parquet(p) if not p.endswith(".csv") else pd.read_csv(p) for p in expanded]
        elif isinstance(src, pd.DataFrame):
            host = [src]
        elif isinstance(src, DeviceFrame):
            return [src]
        elif isinstance(src, dict):
            return [DeviceFrame.from_dict(src, self._device)]
        elif isinstance(src, (list, tuple)):
            out = []
            for s in src:
                out += Dataset(s, device=self._device)._ingest()
            return out
        elif hasattr(src, "to_pandas"):          # pyarrow.Table and friends
            host = [src.to_pandas()]
        else:
            raise TypeError(f"cannot build a Dataset from {type(src)}")
        if self._npartitions and self._npartitions > 1 and len(host) == 1:
            df = host[0]
            n = len(df)
            k = self._npartitions
            # dask's from_pandas split: chunks of ceil(n / k) rows
            chunk = -(-n // k) if n else 0
            host = [df.iloc[i:i + chunk] for i in range(0, n, chunk)] if chunk else [df]
        return [DeviceFrame.from_pandas(h.reset_index(drop=True), self._device) for h in host]

    def _ingest_parquet(self, paths) -> List[DeviceFrame]:
        """Parquet -> partitions without pandas: one partition per row group (or per
        `part_size` rows), decoded by pyarrow straight into data + validity-bitmask buffers
        (nullable int32 stays int32) in pinned host memory; `partitions()` then uploads them
        one ahead of the consumer.  Replaces merlin.io.Dataset(path, engine="parquet",
        part_size=...) (SURVEY.md 8f-1)."""
        import pyarrow as pa
        import pyarrow.parquet as pq
        pin = torch.cuda.is_available()
        rows_per_part = self._part_rows
        parts: List[DeviceFrame] = []
        for p in paths:
            f = pq.ParquetFile(p)
            pending, pending_rows = [], 0

            def flush():
                nonlocal pending, pending_rows
                if pending:
                    parts.append(DeviceFrame.from_arrow(pa.concat_tables(pending), self._device, pin))
                pending, pending_rows = [], 0

            for rg in range(f.num_row_groups):
                t = f.read_row_group(rg)
                if rows_per_part is None:
                    parts.append(DeviceFrame.from_arrow(t, self._device, pin))
                    continue
                while len(t):
                    take = min(len(t), rows_per_part - pending_rows)
                    pending.append(t.slice(0, take))
                    pending_rows += take
                    t = t.slice(take)
                    if pending_rows == rows_per_part:
                        flush()
            flush()
            if f.num_row_groups == 0:
                parts.append(DeviceFrame.from_arrow(f.schema_arrow.empty_table(), self._device, pin))
        if self._npartitions and self._npartitions > 1 and len(parts) == 1 and len(parts[0]):
            whole, n, k = parts[0], len(parts[0]), self._npartitions
            chunk = ((-(-n // k)) + 63) // 64 * 64
            parts = [whole.slice_rows(s0, min(n, s0 + chunk)) for s0 in range(0, n, chunk)]
        return parts

    def partitions(self) -> Iterable[DeviceFrame]:
        """Device-resident partitions, in order.  Partitions that live in (pinned) host
        memory are uploaded on a side stream ONE PARTITION AHEAD of the consumer, so the
        H2D copy of partition i+1 overlaps the kernels working on partition i; uploaded
        partitions stay cached in HBM (a later pass — transform after fit — does not pay
        the copy again) unless `cache_on_device=False`."""
        if self._parts is None:
            self._parts = self._ingest()
        parts = self._parts
        if not any(p.is_host for p in parts) or not torch.cuda.is_available():
            for p in parts:
                yield self._transform(p) if self._transform is not None else p
            return
        dev = torch.device("cuda", torch.cuda.current_device())
        copy_stream = _copy_stream(dev)
        main = torch.cuda.current_stream(dev)
        pending = {}

        def upload(i):
            if i < len(parts) and parts[i].is_host and i not in pending:
                with torch.cuda.stream(copy_stream):
                    d = parts[i].to(dev, non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                self.h2d_bytes += parts[i].nbytes()
                pending[i] = (d, ev)

        upload(0)
        for i in range(len(parts)):
            upload(i + 1)
            if i in pending:
                d, ev = pending.pop(i)
                main.wait_event(ev)
                for c in d._cols.values():          # the consumer stream now owns the buffers
                    c.data.record_stream(main)
                    if c.validity is not None:
                        c.validity.record_stream(main)
                    if c.offsets is not None:
                        c.offsets.record_stream(main)
                if self.cache_on_device:
                    parts[i] = d
                p = d
            else:
                p = parts[i]
            yield self._transform(p) if self._transform is not None else p

    def to_host(self, out: Optional[List[DeviceFrame]] = None) -> List[DeviceFrame]:
        """Materialise every (lazily transformed) partition into pinned host memory.  The
        D2H copy of partition i runs on a side stream while partition i+1 is computed."""
        dev = torch.device("cuda", torch.cuda.current_device())
        out_stream = _copy_stream(dev, 1)
        main = torch.cuda.current_stream(dev)
        # drain what is queued (the tail of a fit) before the D2H pipeline starts: measured on
        # B200, the same fit + transform + to_host step takes ~610 ms with this sync and
        # 760-1370 ms without it (bench.py e2e leg, 2^26 rows; the pipeline below then competes
        # with the fit's still-pending uploads and frees for allocator blocks)
        main.synchronize()
        res: List[DeviceFrame] = []
        for i, part in enumerate(self.partitions()):
            ev = torch.cuda.Event()
            ev.record(main)
            host = out[i] if out is not None and i < len(out) else None
            cols = {}
            with torch.cuda.stream(out_stream):
                out_stream.wait_event(ev)
                for name, c in part.items():
                    hb = host[name].data if host is not None and name in host and \
                        host[name].data.shape == c.data.shape and host[name].data.dtype == c.data.dtype else \
                        torch.empty(c.data.shape, dtype=c.data.dtype, pin_memory=True)
                    hb.copy_(c.data, non_blocking=True)
                    c.data.record_stream(out_stream)
                    hv = None
                    if c.validity is not None:
                        hv = torch.empty(c.validity.shape, dtype=torch.uint8, pin_memory=True)
                        hv.copy_(c.validity, non_blocking=True)
                        c.validity.record_stream(out_stream)
                    hc = Column(hb, hv, c.offsets.cpu() if c.offsets is not None else None,
                                c.dictionary, None, c.is_bool)
                    hc.prehashed = c.prehashed
                    cols[name] = hc
                    self.d2h_bytes += hb.numel() * hb.element_size()
            res.append(DeviceFrame(cols))
        out_stream.synchronize()
        return res

    @property
    def npartitions(self):
        if self._parts is None:
            self._parts = self._ingest()
        return len(self._parts)

    @property
    def num_rows(self):
        if self._parts is None:
            self._parts = self._ingest()
        return sum(len(p) for p in self._parts)

    @property
    def schema(self) -> Schema:
        if self._schema is None:
            if self._parts is None:
                self._parts = self._ingest()
            first = self._parts[0] if self._parts else DeviceFrame()
            if self._transform is not None:
                first = self._transform(first)
            self._schema = _schema_of(first)
        return self._schema

    # ------------------------------------------------------------------ egress
    def to_ddf(self, columns=None, **kwargs) -> _Lazy:
        return _Lazy(self, columns)

    def compute(self, **kwargs) -> pd.DataFrame:
        return self.to_ddf().compute()

    def to_cpu(self):
        self.cpu = True
        return self

    def shuffle_by_keys(self, keys, npartitions: Optional[int] = None) -> "Dataset":
        """A Dataset whose partitions each hold every row of the key tuples they contain: what
        Groupby needs (its transform never moves rows between partitions, reference
        nvtabular/ops/groupby.py:30-35; merlin.io.Dataset.shuffle_by_keys).  Row r goes to
        partition hash(keys of r) % npartitions (default: the current count), with the value hash
        of HashBucket; inside a partition rows keep their order (input partition, then row), so ties
        in Groupby's sort columns resolve as on one partition.  Within one process only."""
        from .dist import world
        from .ops.fill import materialize
        from . import engine
        if world()[0] > 1:
            raise NotImplementedError("shuffle_by_keys moves rows within one process only; under "
                                      "torch.distributed each rank's files must already hold whole key groups")
        keys = [keys] if isinstance(keys, str) else list(keys)
        parts = [DeviceFrame({k: materialize(c) for k, c in p.items()}) for p in self.partitions()]
        k = int(npartitions or len(parts) or 1)
        whole = _concat_frames(parts)
        if not len(whole):
            return Dataset([whole], device=self._device)
        dest = engine.hash_bucket([whole[c] for c in keys], k)
        perm, _ = engine.sort_rows([Column(dest)])
        counts = torch.bincount(dest.long(), minlength=k).tolist()
        out, start = [], 0
        for c in counts:
            p = perm[start:start + c]
            start += c
            cols = {}
            for name, col in whole.items():
                if col.is_list:
                    cols[name] = engine.list_slice(col, 0, np.iinfo(np.int64).max, perm=p, n_rows=c)
                else:
                    cols[name] = engine.gather_rows(col, p, c)
            out.append(DeviceFrame(cols))
        return Dataset(out, device=self._device)

    def to_parquet(self, output_path, shuffle=None, out_files_per_proc=None, seed=None, **kwargs):
        """Write the (lazily transformed) dataset as parquet part files — merlin.io.Dataset.to_parquet
        as the reference's benchmark calls it (bench/examples/dask-nvtabular-criteo-benchmark.py:225-237;
        semantics bench/examples/MultiGPUBench.md:75-89):

          shuffle=None | False        one file per partition, rows in input order
          shuffle="PER_PARTITION"     the rows of every partition are permuted on the device
                                      (torch.randperm + one gather per column) before the D2H copy
          shuffle="PER_WORKER"        every row goes to one of `out_files_per_proc` files of this
                                      process (uniformly at random) and each file is permuted as a
                                      whole when it is closed: the shuffle across partitions that the
                                      reference's per-worker writer cache (nvtabular/worker.py) does

        Under torch.distributed every rank writes its own files (`part_<rank>_<i>.parquet`)."""
        import pyarrow as pa
        import pyarrow.parquet as pq
        from .dist import world
        os.makedirs(output_path, exist_ok=True)
        mode = getattr(shuffle, "name", shuffle)
        mode = str(mode).upper() if mode not in (None, False) else None
        if mode not in (None, "PER_PARTITION", "PER_WORKER", "FULL"):
            raise ValueError(f"unknown shuffle mode {shuffle!r}")
        w, rank = world()
        prefix = f"part_{rank}_" if w > 1 else "part_"
        gen = None
        if mode is not None and torch.cuda.is_available():
            gen = torch.Generator(device="cuda")
            gen.manual_seed(int(seed if seed is not None else 0x5EED) + rank)
        if mode in (None, "PER_PARTITION"):
            for i, part in enumerate(self.partitions()):
                if mode == "PER_PARTITION" and len(part):
                    part = _permute_rows(part, torch.randperm(len(part), generator=gen, device="cuda"))
                pq.write_table(part.to_arrow(), os.path.join(output_path, f"{prefix}{i}.parquet"))
            return output_path
        nfiles = int(out_files_per_proc or 1)
        buckets = [[] for _ in range(nfiles)]
        for part in self.partitions():
            n = len(part)
            if n == 0:
                continue
            dest = torch.randint(0, nfiles, (n,), generator=gen, device="cuda")
            order = torch.argsort(dest, stable=True)
            counts = torch.bincount(dest, minlength=nfiles).cpu().tolist()
            tab = _permute_rows(part, order).to_arrow()
            off = 0
            for f, c in enumerate(counts):
                if c:
                    buckets[f].append(tab.slice(off, c))
                off += c
        rng = np.random.default_rng(int(seed if seed is not None else 0x5EED) + 7919 * (rank + 1))
        for f, chunks in enumerate(buckets):
            if not chunks:
                continue
            tab = pa.concat_tables(chunks)
            tab = tab.take(pa.array(rng.permutation(len(tab))))
            pq.write_table(tab, os.path.join(output_path, f"{prefix}{f}.parquet"))
        return output_path


def _concat_columns(cols: List[Column]) -> Column:
    """rows of several columns one after the other; string dictionaries are merged (codes stay
    order-preserving) and list offsets rebased"""
    from .column import pack_validity, unpack_validity
    if len(cols) == 1:
        return cols[0]
    dictionary = None
    datas = [c.data for c in cols]
    if any(c.dictionary is not None for c in cols):
        dictionary = np.array(sorted(set().union(*[set(c.dictionary.tolist()) for c in cols
                                                   if c.dictionary is not None])), dtype=object)
        datas = []
        for c in cols:
            if c.dictionary is None or not len(c.dictionary):
                datas.append(torch.zeros_like(c.data))
                continue
            lut = torch.from_numpy(np.searchsorted(dictionary, c.dictionary).astype(np.int32)).to(c.data.device)
            datas.append(lut[c.data.long()])
    validity = None
    if any(c.validity is not None for c in cols):
        validity = pack_validity(torch.cat([unpack_validity(c.validity, c.data.numel(), c.data.device) for c in cols]))
    offsets = None
    if cols[0].offsets is not None:
        pieces, base = [], 0
        for c in cols:
            pieces.append(c.offsets[:-1] + base)
            base += int(c.data.numel())
        pieces.append(torch.tensor([base], dtype=torch.int64, device=cols[0].data.device))
        offsets = torch.cat(pieces)
    return Column(torch.cat(datas), validity, offsets, dictionary, None, cols[0].is_bool)


def _concat_frames(frames: List[DeviceFrame]) -> DeviceFrame:
    if not frames:
        return DeviceFrame()
    return DeviceFrame({name: _concat_columns([f[name] for f in frames]) for name in frames[0].columns})


def _permute_rows(frame: DeviceFrame, perm: torch.Tensor) -> DeviceFrame:
    """frame[perm] for flat columns (data + validity); list columns are not shuffled row-wise here"""
    from .column import pack_validity, unpack_validity
    out = {}
    n = len(frame)
    for name, c in frame.items():
        if c.offsets is not None:
            raise NotImplementedError("shuffling list columns")
        from .ops.fill import materialize
        c = materialize(c)
        v = None
        if c.validity is not None:
            v = pack_validity(unpack_validity(c.validity, n)[perm])
        col = Column(c.data[perm], v, None, c.dictionary, None, c.is_bool)
        col.prehashed = c.prehashed
        out[name] = col
    return DeviceFrame(out)
