#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on synthetic tables, this repo's engine or the
reference's CPU path (oracle port) beside it.

    python bench.py --gpus N --steps K --warmup W                 # configs[1]/[2]: Criteo-1TB-shaped
    python bench.py --workload hashbucket ...                      # configs[4]: HashBucket 40 x int64
    python bench.py --workload movielens ...                       # configs[3]: JoinGroupby + TargetEncoding
    python bench.py --impl reference [--workload ...] ...          # the reference's CPU path, all host cores
    python bench.py ... --dump-outputs DIR                         # + the last timed step's outputs, sampled

Default workload (criteo): a "step" = Workflow.fit(dataset) + Workflow.transform(dataset) over the
whole HBM-resident table of 2.5e8 rows per GPU (SURVEY.md 8d C2), categorical cardinalities of the
full 4.37e9-row Criteo-1TB profile, fit accumulated over the table's partitions, outputs produced
partition by partition.  Prints ONE JSON line: `value` = device-resident throughput, `e2e` = the same
workflow fed from pinned HOST buffers with the H2D / D2H copies inside the timed region, `roofline`
= the dominant kernel family against the measured HBM peak, `cpu_baseline` = the CPU oracle timed on
this box, `parity_gate` = what was checked on this very process group before anything was timed.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES = {           # SURVEY.md 8d, algorithmic bytes per row
    "criteo": 641.75,            # fit 160.875 + transform 480.875 (int64 labels, float64 conts)
    "criteo32": 485.75,          # 32-bit outputs
    "hashbucket": 480.0,         # 40 columns x (8 read + 4 written)
    "movielens": 84.0,           # fit 12 + transform 12 read + 60 written
}
METRIC = {
    "criteo": "rows/sec Criteo-1TB-shaped Categorify+FillMissing+Normalize",
    "hashbucket": "rows/sec HashBucket(2^20) over 40 int64 key columns",
    "movielens": "rows/sec MovieLens-shaped JoinGroupby+TargetEncoding",
}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _traffic(workload, kernel, rows):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel family from
    the committed ncu capture (profiles/traffic_r2.json, tools/summarize_ncu.py); only valid for
    the workload and row count it was captured at, null otherwise."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_r2.json")) as f:
            d = json.load(f)
        e = d.get(workload, {}).get(kernel)
        if e and int(e.get("rows_per_gpu", -1)) == int(rows):
            return float(e["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def _host_memory_budget():
    """bytes of host memory this container may still take: the cgroup limit (v2, then v1) minus its
    current charge, capped by MemAvailable.  None when nothing can be read."""
    def _read_int(path):
        try:
            v = open(path).read().strip()
            return None if v == "max" else int(v)
        except Exception:
            return None
    cands = []
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        limit = _read_int(lim)
        if limit is not None and limit < (1 << 60):
            cands.append(limit - (_read_int(cur) or 0))
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                cands.append(int(ln.split()[1]) * 1024)
    except Exception:
        pass
    return min(cands) if cands else None


def e2e_rows_within_host_memory(want_rows, bytes_per_row, local_ranks, budget):
    """The e2e leg pins its inputs AND its results (bytes_per_row of both per row) in every rank of
    the box; a pinned page is charged to the container, and a container over its limit is killed,
    not refused.  Keep the ranks' sum below 80 % of `budget`; whole 2^23-row partitions (their pinned
    buffers are exact powers of two), at least one.  `budget` None = unknown = leave the request."""
    if budget is None:
        return want_rows
    fit = int(budget * 0.8 / max(local_ranks, 1) / bytes_per_row)
    if fit >= want_rows:
        return want_rows
    return max(1 << 23, fit >> 23 << 23)



E2E_PINNED_BYTES_PER_ROW = 512      # measured: 480.6 (profiles/bench_r2_criteo_1gpu.json: (h2d + d2h) / rows)


def _cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _bind_to_gpu_numa_node(local_rank):
    """Run this rank's host threads (and first-touch its pinned buffers) on the NUMA node its GPU
    hangs off: with 8 ranks on a two-socket host the e2e leg otherwise crosses the socket link for
    half of the GPUs.  Best effort."""
    try:
        import torch
        bdf = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bdf, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = []
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids)
        return node
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  ONE nvidia-smi
    process, started before the warm-up (its start-up takes driver-wide locks for hundreds
    of ms and would otherwise land inside a short timed region) and left polling every
    50 ms; stop(t0, t1) keeps the samples whose own timestamps fall inside the region."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                 os.environ.get("NVTB_SMI_MS", "50"), "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    @staticmethod
    def _epoch(stamp):
        import datetime
        try:
            return datetime.datetime.strptime(stamp.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 10:
                continue
            try:
                rows.append((self._epoch(f[0]), float(f[2]), float(f[3]), f[6:10]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 is not None and r[0] is not None and t0 - 0.05 <= r[0] <= t1 + 0.05]
        window = "timed region"
        if not inside:          # region shorter than the polling period: nearest samples
            inside, window = rows[-3:], "nearest samples (region shorter than the 50 ms poll)"
        sm, mx, reasons = [r[1] for r in inside], [r[2] for r in inside], set()
        for r in inside:
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# =======================================================================================
# workloads: every one provides make_table / build_workflow / step / e2e pieces
# =======================================================================================
def cut(frame, nparts):
    """the resident table cut into `nparts` row partitions (views, 64-row aligned)"""
    rows = len(frame)
    chunk = ((rows + nparts - 1) // nparts + 63) // 64 * 64
    return [frame.slice_rows(s, min(rows, s + chunk)) for s in range(0, rows, chunk)]


def build_workflow(nvt, workload, out_path, int32_outputs=False):
    ops = nvt.ops
    if workload == "criteo":
        from nvtabular_b200.synth import CAT_NAMES, CONT_NAMES
        cat_kw = {"dtype": "int32"} if int32_outputs else {}
        norm_kw = {"out_dtype": "float32"} if int32_outputs else {}
        cats = CAT_NAMES >> ops.Categorify(out_path=out_path, **cat_kw)
        conts = CONT_NAMES >> ops.FillMissing() >> ops.Normalize(**norm_kw)
        return nvt.Workflow(cats + conts + ["label"])
    if workload == "hashbucket":
        return nvt.Workflow([f"K{j + 1}" for j in range(40)] >> ops.HashBucket(1 << 20))
    if workload == "movielens":
        groups = ["userId", "movieId", ["userId", "movieId"]]
        jg = groups >> ops.JoinGroupby(out_path=out_path, cont_cols=["rating"], stats=["count", "sum", "mean", "std"])
        te = groups >> ops.TargetEncoding("rating", kfold=5, p_smooth=20, out_path=out_path)
        return nvt.Workflow(jg + te)
    raise ValueError(workload)


def make_table(workload, rows, device, rank, profile_rows):
    from nvtabular_b200 import synth
    if workload == "criteo":
        return synth.criteo_frame(rows, total_rows=profile_rows, device=device, rank=rank)
    if workload == "hashbucket":
        return synth.hashbucket_frame(rows, 40, device=device, rank=rank)
    return synth.movielens_frame(rows, device=device, rank=rank)


def run_step(nvt, wf, parts, fit=True, sink=None):
    """one pass of the hot path over the resident table: fit (accumulated over the partitions,
    artefact files written — Workflow.fit joins its writer threads), then transform partition
    by partition (the outputs of one partition live at a time; `sink(i, part)` sees each)"""
    ds = nvt.Dataset(list(parts))
    if fit:
        wf.fit(ds)
    out = None
    for i, part in enumerate(wf.transform(ds).partitions()):
        if sink is not None:
            sink(i, part)
        out = part
    return out


DUMP_BYTES = 64 << 20        # --dump-outputs writes at most this much
DUMP_ROWS = 1 << 17


class OutputSample:
    """--dump-outputs: the same seeded sample of rows of every output column of one step.
    take(i, part) gathers the sampled rows of output partition i on the device while the step
    runs (a step keeps one partition's outputs alive at a time); save(dir) writes <column>.npy
    and row_index.npy (the sampled rows of the table).  Float32 columns stay float32, all other
    columns become float64 (integers below 2^53 exactly), nulls become NaN."""

    def __init__(self, part_rows, ncols, device, seed=0):
        import numpy as np
        import torch
        total = sum(part_rows)
        n = min(total, DUMP_ROWS, DUMP_BYTES // (8 * (ncols + 1)))
        self.rows = np.sort(np.random.default_rng(seed).choice(total, size=n, replace=False))
        self.part_rows = list(part_rows)
        bounds = np.cumsum([0] + self.part_rows)
        self.local = [torch.from_numpy(self.rows[(self.rows >= s) & (self.rows < e)] - s).to(device)
                      for s, e in zip(bounds[:-1], bounds[1:])]
        self.parts = [None] * len(self.part_rows)

    def take(self, i, part):
        import torch
        if len(part) != self.part_rows[i]:
            raise ValueError(f"output partition {i} has {len(part)} rows, its input {self.part_rows[i]}")
        idx, got = self.local[i], {}
        for name, col in part.items():
            if col.offsets is not None:
                raise ValueError(f"--dump-outputs: list column {name} is not supported")
            valid = None
            if col.validity is not None:      # Arrow bitmask: bit (r & 7) of byte (r >> 3)
                valid = (col.validity.index_select(0, idx >> 3) >> (idx & 7).to(torch.uint8)) & 1
            got[name] = (col.data.index_select(0, idx), valid)
        self.parts[i] = got

    def save(self, out_dir):
        import numpy as np
        import torch
        if any(p is None for p in self.parts):
            raise RuntimeError("--dump-outputs: the timed step did not produce every partition")
        arrays = {"row_index": self.rows.astype(np.float64)}
        for name in self.parts[0]:
            if name in arrays:
                raise ValueError(f"--dump-outputs: output column {name} clashes with row_index.npy")
            vals = torch.cat([p[name][0] for p in self.parts]).cpu().numpy()
            if vals.dtype.kind in "iu" and vals.size and np.abs(vals.astype(np.float64)).max() >= 2.0 ** 53:
                raise ValueError(f"--dump-outputs: integer column {name} is not exact in float64")
            out = vals.astype(np.float32 if vals.dtype == np.float32 else np.float64)
            valid = [np.ones(len(d), bool) if v is None else v.cpu().numpy() == 1
                     for d, v in (p[name] for p in self.parts)]
            out[~np.concatenate(valid)] = np.nan
            arrays[name] = out
        total = sum(a.nbytes for a in arrays.values())
        if total > DUMP_BYTES:
            raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)
        return sorted(arrays), total


def host_partitions(frame, nparts):
    """pinned-host mirror of a device frame, cut into `nparts` row partitions"""
    return [p.pin() for p in cut(frame, nparts)]


def run_step_e2e(nvt, wf, host_parts, out_host, fit=True):
    """The same step from HOST buffers through the public API: Dataset of pinned host
    partitions -> Workflow.fit -> Workflow.transform -> pinned host results.  Every input
    byte crosses PCIe once (partitions are prefetched one ahead and stay in HBM between
    fit and transform), every output byte crosses it once (D2H overlapped with the next
    partition's kernels)."""
    trace = os.environ.get("NVTB_BENCH_DUMP")
    t0 = time.perf_counter()
    ds = nvt.Dataset(list(host_parts))
    if fit:
        wf.fit(ds)
    if trace:
        import torch
        torch.cuda.synchronize()
        t1 = time.perf_counter()
    tds = wf.transform(ds)
    res = tds.to_host(out_host if out_host else None)
    if trace:
        ms = torch.cuda.memory_stats()
        sys.stderr.write("[bench dump] e2e step: fit %.1f ms, transform+to_host %.1f ms; cudaMalloc %d cudaFree %d "
                         "retries %d reserved %.1f GB\n"
                         % ((t1 - t0) * 1e3, (time.perf_counter() - t1) * 1e3, ms.get("num_device_alloc", -1),
                            ms.get("num_device_free", -1), ms.get("num_alloc_retries", -1),
                            ms.get("reserved_bytes.all.current", 0) / 1e9))
    return ds.h2d_bytes, tds.d2h_bytes, res


# =======================================================================================
# CPU reference (oracle port): bounded samples of the same workloads
# =======================================================================================
def cpu_reference(workload, rows, workers, profile_rows, steps=1, warmup=0, budget_s=None):
    """The reference's CPU path (oracle/parallel.py) on a bounded sample of the same synthetic
    workload, generated with the same generator code on the CPU.  With `budget_s` the sample is
    SIZED so that warmup + steps passes fit the budget: a calibration pass over the first 2^18 rows
    gives the rate, the sample is the first min(rows, rate x budget per step / 2) rows (the /2
    covers the super-linear merge of the partials).  -> (rows/s, seconds per step, steps run,
    rows per step)"""
    from nvtabular_b200 import synth
    if workload == "criteo":
        from oracle.parallel import run_criteo_workflow
        frame = synth.criteo_frame(rows, total_rows=profile_rows, device="cpu")
        df = synth.frame_to_pandas_nullable(frame)
        # what pandas itself holds for a nullable int column read from parquet: float64 + NaN
        df = df.astype({c: "float64" for c in synth.CAT_NAMES + synth.CONT_NAMES})

        def once(n):
            tf, tt, *_ = run_criteo_workflow(df.iloc[:n], synth.CAT_NAMES, synth.CONT_NAMES, workers)
            return tf + tt
    elif workload == "hashbucket":
        from oracle.parallel import run_hashbucket
        frame = synth.hashbucket_frame(rows, 40, device="cpu")
        cols = [frame[c].data.numpy() for c in frame.columns]

        def once(n):
            return run_hashbucket([c[:n] for c in cols], 1 << 20, workers)
    else:
        from oracle.parallel import run_movielens_workflow
        frame = synth.movielens_frame(rows, device="cpu")
        df = frame.to_pandas()

        def once(n):
            tf, tt = run_movielens_workflow(df.iloc[:n].reset_index(drop=True), workers)
            return tf + tt
    n_step = rows
    if budget_s is not None:
        n_cal = min(rows, 1 << 18)
        t_cal = max(once(n_cal), 1e-3)
        per_step = budget_s / max(1, steps + warmup)
        n_step = int(min(rows, max(n_cal, (n_cal / t_cal) * per_step * 0.5)))
    times = []
    for i in range(warmup + steps):
        t = once(n_step)
        if i >= warmup:
            times.append(t)
    sec = sum(times) / len(times)
    return n_step / sec, sec, len(times), n_step


CPU_SAMPLE_ROWS = {"criteo": (1 << 20, 1 << 22), "hashbucket": (1 << 20, 1 << 23), "movielens": (1 << 20, 1 << 23)}


def workload_config(args, world, rows):
    total = rows * world
    if args.workload == "criteo":
        which = "configs[1]" if world == 1 else f"configs[2] (the configs[1] workflow sharded over {world} B200s)"
        return {"workload": f"BASELINE.json {which}: Criteo-1TB-shaped synthetic (13 int + 26 cat int32, "
                            "nullable), Categorify+FillMissing+Normalize, one step = Workflow.fit + "
                            "Workflow.transform over the HBM-resident table",
                "rows_per_gpu": rows, "total_rows": total, "partitions_per_gpu": args.parts,
                "cardinality_profile_rows": args.profile_rows,
                "outputs": "int32 labels, float32 conts" if args.int32_outputs else "int64 labels, float64 conts",
                "algorithmic_bytes_per_row": ALGO_BYTES["criteo32" if args.int32_outputs else "criteo"],
                "cache": "inputs (%.1f GB/GPU) larger than L2; no explicit flush" % (rows * 160.9 / 1e9),
                "artifacts": {"eager": "library default: every meta.<col>.parquet and the unique.<col>.parquet of "
                                       "every vocabulary up to 2^20 keys written inside fit (under the GPU's "
                                       "builds of the large vocabularies); larger vocabulary files on first read",
                              "lazy": "deferred until read"}[args.artifacts],
                "parallelism": (f"row-sharded x{world}; NCCL: moments all-reduce, key-hash owner merge (small "
                                f"columns), key-range exchange of sorted pairs + shard all-gather (large columns)")
                if world > 1 else "single GPU"}
    if args.workload == "hashbucket":
        return {"workload": "BASELINE.json configs[4]: 40 int64 key columns, keys uniform over 1e8 ids through a "
                            "64-bit bijection, HashBucket(num_buckets=2**20), one step = Workflow.transform over "
                            "the HBM-resident table",
                "rows_per_gpu": rows, "total_rows": total, "partitions_per_gpu": args.parts,
                "outputs": "int32 buckets", "algorithmic_bytes_per_row": ALGO_BYTES["hashbucket"],
                "cache": "inputs (%.1f GB/GPU) larger than L2; no explicit flush" % (rows * 320 / 1e9),
                "parallelism": f"row-sharded x{world}, no exchange" if world > 1 else "single GPU"}
    return {"workload": "BASELINE.json configs[3]: MovieLens-shaped ratings (userId K=1.6e5, movieId K=6e4, rating "
                        "float32), [userId, movieId, (userId, movieId)] >> JoinGroupby(rating: count,sum,mean,std) + "
                        "TargetEncoding(rating, kfold=5, p_smooth=20), one step = Workflow.fit + Workflow.transform",
            "rows_per_gpu": rows, "total_rows": total, "partitions_per_gpu": args.parts,
            "outputs": "float32 stats, int32 counts, float32 TE", "algorithmic_bytes_per_row": ALGO_BYTES["movielens"],
            "cache": "inputs (%.2f GB/GPU) larger than L2; no explicit flush" % (rows * 12 / 1e9),
            "parallelism": f"row-sharded x{world}, key-hash owner merge over NCCL" if world > 1 else "single GPU"}


# =======================================================================================
# parity gate: run before anything is timed, on the process group that is about to be timed
# =======================================================================================
def _digest(tensors):
    h = hashlib.sha1()
    for t in tensors:
        h.update(t.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()[:16]


def _same_state(a, b):
    if set(a) != set(b):
        return False
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, list) and isinstance(y, list):
            if len(x) != len(y) or any(abs(p - q) > 1e-9 * max(1.0, abs(p), abs(q)) for p, q in zip(x, y)):
                return False
        elif x != y:
            return False
    return True


def parity_gate(nvt, workload, rank, world, dev, tmp_root):
    """A small seeded table (every rank a different shard) through the SAME code paths the timed
    run takes (NVTB_RUNS_MIN_KEYS lowered so that the sorted accumulator is exercised):
      1. the fitted state (vocabulary keys / sizes / null counts, means / stds, group tables) of
         the N-rank fit is identical on every rank and equals a single-process fit of the union
         of the shards on this very GPU;
      2. on rank 0, labels / buckets / statistics of a sample equal an independent pandas / numpy
         computation over the union (value_counts + (count desc, key asc) order; pandas value
         hash; groupby sums).
    Returns a dict for the JSON line; raises on a mismatch."""
    import numpy as np
    import pandas as pd
    import torch
    import torch.distributed as dist
    from nvtabular_b200 import synth
    from nvtabular_b200.column import Column, DeviceFrame, unpack_validity
    t0 = time.perf_counter()
    rows = 1 << 19
    old_env = os.environ.get("NVTB_RUNS_MIN_KEYS")
    os.environ["NVTB_RUNS_MIN_KEYS"] = "200000"
    checks = []
    try:
        if workload == "criteo":
            local = synth.criteo_frame(rows, total_rows=40_000_000, device=dev, rank=rank, seed=4242)
        elif workload == "hashbucket":
            local = synth.hashbucket_frame(rows, 40, device=dev, rank=rank, seed=4242)
        else:
            local = synth.movielens_frame(rows, device=dev, rank=rank, seed=4242)

        def gather_union():
            if world == 1:
                return local
            cols = {}
            for name, c in local.items():
                parts = [torch.empty_like(c.data) for _ in range(world)]
                dist.all_gather(parts, c.data.contiguous())
                data = torch.cat(parts)
                val = None
                if c.validity is not None:
                    v = unpack_validity(c.validity, rows).to(torch.uint8)
                    vp = [torch.empty_like(v) for _ in range(world)]
                    dist.all_gather(vp, v)
                    from nvtabular_b200.column import pack_validity
                    val = pack_validity(torch.cat(vp).bool())
                cols[name] = Column(data, val)
            return DeviceFrame(cols)

        def state_of(wf):
            out = {}
            for n in wf.output_node.topo_order():
                if n.kind != "op":
                    continue
                op = n.op
                if hasattr(op, "categories") and hasattr(op.categories, "fitted"):
                    for name, fv in op.categories.fitted.items():
                        k, s = fv.vocab.export()
                        out["cat." + name] = _digest([k, s]) + ":%d:%d" % (fv.vocab.null_size, fv.vocab.n_kept)
                if hasattr(op, "means") and isinstance(getattr(op, "means"), dict):
                    out["means"] = repr(sorted((k, float(v)) for k, v in op.means.items()))
                if hasattr(op, "stds") and isinstance(getattr(op, "stds"), dict):
                    out["stds"] = repr(sorted((k, float(v)) for k, v in op.stds.items()))
                if hasattr(op, "tables") and isinstance(getattr(op, "tables"), dict):
                    for name, tb in op.tables.items():
                        df = tb.frame() if callable(getattr(tb, "frame", None)) else tb
                        if not isinstance(df, pd.DataFrame):
                            continue
                        keyc = [c for c in df.columns if not (c.startswith(name + "_") or c == name + "_count")]
                        df = df.sort_values(keyc).reset_index(drop=True)
                        exact = [c for c in df.columns if c in keyc or c.endswith("_count")]
                        out["jg." + name] = hashlib.sha1(
                            df[exact].to_numpy(dtype="float64").tobytes()).hexdigest()[:16]
                        # floating sums are accumulated with fp64 atomics (order varies): compared at 1e-9
                        out["jgsum." + name] = [float(np.nansum(df[c].to_numpy(dtype="float64")))
                                                for c in df.columns if c not in exact]
            return out

        tmp = os.path.join(tmp_root, "gate")
        wf = build_workflow(nvt, workload, tmp)
        ds = nvt.Dataset(cut(local, 3))
        if workload != "hashbucket":
            wf.fit(ds)
        st = state_of(wf)
        out_local = next(iter(wf.transform(nvt.Dataset(local)).partitions()))
        union = gather_union()
        if world > 1:
            seen = [None] * world
            dist.all_gather_object(seen, st)
            assert all(_same_state(s, seen[0]) for s in seen), "fitted state differs between ranks"
            checks.append(f"fitted state identical on {world} ranks ({len(st)} digests)")
            # single-process fit of the union on this GPU, collectives disabled
            os.environ["NVTB_DISABLE_DIST"] = "1"
            try:
                wf1 = build_workflow(nvt, workload, tmp + "_single")
                if workload != "hashbucket":
                    wf1.fit(nvt.Dataset(cut(union, 2)))
                st1 = state_of(wf1)
            finally:
                os.environ.pop("NVTB_DISABLE_DIST", None)
            bad = [k for k in st1 if not _same_state({k: st.get(k)}, {k: st1[k]})]
            assert not bad and set(st) == set(st1), f"distributed fit != single-process fit of the union: {bad[:4]}"
            checks.append("distributed fit == single-process fit of the union")
        # independent host computation on rank 0
        if rank == 0:
            nsamp = 1 << 15
            if workload == "criteo":
                for c in ["C1", "C6", "C20", "C23"]:
                    col = union[c]
                    valid = unpack_validity(col.validity, len(union)).cpu().numpy() if col.validity is not None \
                        else np.ones(len(union), bool)
                    keys = col.data.cpu().numpy()
                    vc = pd.Series(keys[valid]).value_counts(sort=False)
                    order = pd.DataFrame({"k": vc.index.to_numpy(), "s": vc.to_numpy()}).sort_values(
                        ["s", "k"], ascending=[False, True], kind="stable")
                    pos = pd.Series(np.arange(len(order), dtype=np.int64) + 3, index=order["k"].to_numpy())
                    lk = local[c].data[:nsamp].cpu().numpy()
                    lv = unpack_validity(local[c].validity, rows)[:nsamp].cpu().numpy() \
                        if local[c].validity is not None else np.ones(nsamp, bool)
                    exp = np.where(lv, pos.reindex(lk).to_numpy(), 1)
                    got = out_local[c].data[:nsamp].cpu().numpy()
                    assert np.array_equal(got, exp), f"labels of {c} differ from pandas value_counts order"
                for c in ["I1", "I13"]:
                    col = union[c]
                    valid = unpack_validity(col.validity, len(union)).cpu().numpy() if col.validity is not None \
                        else np.ones(len(union), bool)
                    x = np.where(valid, col.data.cpu().numpy().astype(np.float64), 0.0)
                    mean, std = x.mean(), x.std(ddof=0)
                    lx = local[c].data[:nsamp].cpu().numpy().astype(np.float64)
                    lv = unpack_validity(local[c].validity, rows)[:nsamp].cpu().numpy() \
                        if local[c].validity is not None else np.ones(nsamp, bool)
                    exp = (np.where(lv, lx, 0.0) - mean) / std
                    got = out_local[c].data[:nsamp].cpu().numpy()
                    assert np.allclose(got, exp, rtol=1e-5, atol=1e-9), f"normalised {c} differs (rtol 1e-5)"
                checks.append("rank-0 sample: labels of C1,C6,C20,C23 == pandas order; I1,I13 normalised within 1e-5")
            elif workload == "hashbucket":
                for c in ["K1", "K17", "K40"]:
                    k = local[c].data[:nsamp].cpu().numpy()
                    exp = (pd.util.hash_array(k, categorize=False) % np.uint64(1 << 20)).astype(np.int32)
                    assert np.array_equal(out_local[c].data[:nsamp].cpu().numpy(), exp), f"buckets of {c} differ"
                checks.append("rank-0 sample: buckets of K1,K17,K40 == pandas.util.hash_array % 2^20")
            else:
                u = union.to_pandas()
                g = u.groupby("userId")["rating"].agg(["count", "sum"])
                lk = local["userId"].data[:nsamp].cpu().numpy()
                exp_cnt = g["count"].reindex(lk).to_numpy()
                exp_sum = g["sum"].reindex(lk).to_numpy()
                assert np.array_equal(out_local["userId_count"].data[:nsamp].cpu().numpy(), exp_cnt)
                assert np.allclose(out_local["userId_rating_sum"].data[:nsamp].cpu().numpy(), exp_sum, rtol=1e-6)
                checks.append("rank-0 sample: userId count/sum == pandas groupby over the union")
        if world > 1:
            dist.barrier()
    finally:
        if old_env is None:
            os.environ.pop("NVTB_RUNS_MIN_KEYS", None)
        else:
            os.environ["NVTB_RUNS_MIN_KEYS"] = old_env
    return {"status": "ok", "rows_per_rank": rows, "ranks": world, "checks": checks,
            "seconds": round(time.perf_counter() - t0, 2)}


# =======================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="criteo", choices=["criteo", "hashbucket", "movielens"])
    ap.add_argument("--rows", type=int, default=0,
                    help="rows resident per GPU (default: 2.5e8 criteo / hashbucket — SURVEY 8d C2/C5; 2.5e7 movielens)")
    ap.add_argument("--parts", type=int, default=4, help="device-resident partitions the table is cut into")
    ap.add_argument("--profile-rows", type=int, default=4_370_000_000,
                    help="row count the categorical cardinalities are scaled to (4.37e9 = the full Criteo-1TB profile)")
    ap.add_argument("--e2e-rows", type=int, default=0,
                    help="rows per GPU per e2e step (default: the first min(rows, 2^27) rows of the same table)")
    ap.add_argument("--e2e-parts", type=int, default=0, help="host partitions per e2e step (default: 2^23 rows each)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the bounded CPU sample")
    ap.add_argument("--int32-outputs", action="store_true", help="Categorify(dtype=int32), Normalize(float32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gate", action="store_true", help="skip the parity gate")
    ap.add_argument("--artifacts", default="eager", choices=["eager", "lazy"],
                    help="NVTB_ARTIFACTS for the timed steps (eager = library default)")
    ap.add_argument("--sweep", default="", help="hashbucket: comma-separated row counts for the roofline curve")
    ap.add_argument("--pyprofile", action="store_true", help="cProfile one extra step to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed (rank 0): every output "
                         f"column at the same {DUMP_ROWS} seeded sample rows, as DIR/<column>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    os.environ["NVTB_ARTIFACTS"] = args.artifacts
    args.warmup = max(args.warmup, 0)
    wl = args.workload
    rows = args.rows or {"criteo": 250_000_000, "hashbucket": 250_000_000, "movielens": 25_000_000}[wl]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    # -------------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        cores = os.cpu_count() or 1
        cpu_rows = args.cpu_rows or CPU_SAMPLE_ROWS[wl][1]
        value, sec, ran, cpu_rows = cpu_reference(wl, cpu_rows, cores, args.profile_rows, steps=max(1, args.steps),
                                                  warmup=args.warmup, budget_s=float(os.environ.get("NVTB_REF_BUDGET_S", "150")))
        line = {
            "impl": "reference", "metric": METRIC[wl], "value": value, "unit": "rows/s", "n_gpus": args.gpus,
            "steps": ran, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64" if wl == "criteo" else ("u64" if wl == "hashbucket" else "f64"),
            "data": "synthetic", "config": workload_config(args, world, rows),
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "cpu_model": _cpu_model(),
                             "kind": "port",
                             "sample": f"each step = {'fit+transform' if wl != 'hashbucket' else 'transform'} of the first "
                                       f"{cpu_rows} rows of the same synthetic table (same generator, same cardinality "
                                       f"profile; sized by a calibration pass so that warmup + steps fit "
                                       f"~{os.environ.get('NVTB_REF_BUDGET_S', '150')} s), partition-parallel over "
                                       f"{cores} processes (oracle/parallel.py); {sec:.2f} s per step"},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # -------------------------------------------------------------------- this repo's engine
    import torch
    import torch.distributed as dist
    import nvtabular_b200 as nvt
    from nvtabular_b200 import engine

    torch.cuda.set_device(local_rank)
    numa = _bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    total_rows = rows * world

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # the artefact files of the fits go to a private directory, removed at exit: the source tree
    # may be read-only, and a fixed /tmp name may belong to another user of the machine
    tmp_root = tempfile.TemporaryDirectory(prefix=f"nvtb_bench_rank{rank}_", ignore_cleanup_errors=True)
    gate = {"status": "skipped"}
    if not args.no_gate:
        gate = parity_gate(nvt, wl, rank, world, dev, tmp_root.name)
        torch.cuda.empty_cache()

    table = make_table(wl, rows, dev, rank, args.profile_rows)
    frame = cut(table, args.parts)
    out_dir = os.path.join(tmp_root.name, "bench")
    wf = build_workflow(nvt, wl, out_dir, args.int32_outputs)
    has_fit = wl != "hashbucket"

    # cold first fit of a fresh Workflow: allocations, table sizing, sampling passes included
    first_fit_ms = None
    if has_fit:
        sync_all()
        t0 = time.perf_counter()
        wf.fit(nvt.Dataset(list(frame)))
        torch.cuda.synchronize()
        first_fit_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([first_fit_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            first_fit_ms = float(t.item())

    if args.pyprofile and rank == 0:
        import cProfile
        import pstats
        run_step(nvt, wf, frame, has_fit)
        torch.cuda.synchronize()
        pr = cProfile.Profile()
        pr.enable()
        run_step(nvt, wf, frame, has_fit)
        torch.cuda.synchronize()
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(35)

    def timed(parts, steps, warmup, with_profile=True, sampler=None, sink=None):
        for _ in range(warmup):
            out = run_step(nvt, wf, parts, has_fit)
            del out
        sync_all()
        engine.profile = [] if with_profile else None
        t_wall0 = time.time()
        launches0 = engine.kernel_launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            out = run_step(nvt, wf, parts, has_fit, sink if i == steps - 1 else None)
            del out
        ev1.record()
        sync_all()
        prof = engine.profile or []
        engine.profile = None
        clocks = sampler.stop(t_wall0, time.time()) if sampler is not None else None
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, engine.kernel_launches - launches0, prof, clocks

    # ---------------- device-resident timing --------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_sampler = time.time()
    if sampler:
        sampler.start()
    for _ in range(min(1, args.warmup)):          # the first warm-up step before the sampler's settle wait
        out = run_step(nvt, wf, frame, has_fit)
        del out
    if rank == 0 and time.time() - t_sampler < 1.5:      # nvidia-smi start-up must be over
        time.sleep(1.5 - (time.time() - t_sampler))
    dump = None
    if args.dump_outputs and rank == 0:
        dump = OutputSample([len(p) for p in frame], len(wf.output_node.output_columns.names), dev)
    ms_per_step, launches, prof, clocks = timed(frame, args.steps, max(0, args.warmup - 1), True, sampler,
                                                dump.take if dump else None)
    value = total_rows / (ms_per_step / 1e3)
    if dump:
        names, nbytes = dump.save(args.dump_outputs)
        sys.stderr.write(f"[bench] last timed step: {len(dump.rows)} sampled rows of {len(names) - 1} output "
                         f"columns ({nbytes} bytes) written to {args.dump_outputs}\n")
        dump = None

    # per-kernel-family device time (CUDA events on the launching stream)
    fam = {}
    for family, s, e, nbytes in prof:
        d = fam.setdefault(family, {"ms": 0.0, "bytes": 0.0, "launches": 0})
        d["ms"] += s.elapsed_time(e)
        d["bytes"] += nbytes
        d["launches"] += 1
    if os.environ.get("NVTB_BENCH_DUMP") and rank == 0:
        per_step = len(prof) // max(1, args.steps)
        for st in range(args.steps):
            sys.stderr.write("[bench dump] step %d: %s\n" % (st, " ".join(
                "%s:%.0f" % (f[:3] + f[-3:], s.elapsed_time(e) * 1e3)
                for f, s, e, _ in prof[st * per_step:(st + 1) * per_step])))
    peak, peak_src = _peaks()
    algo = ALGO_BYTES["criteo32"] if (wl == "criteo" and args.int32_outputs) else ALGO_BYTES[wl]
    kernels = {}
    for k, d in fam.items():
        gbs = d["bytes"] / (d["ms"] / 1e3) / 1e9 if d["ms"] > 0 else 0.0
        kernels[k] = {"ms_per_step": d["ms"] / args.steps, "launches_per_step": d["launches"] / args.steps,
                      "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
    dominant = max(fam, key=lambda k: fam[k]["ms"]) if fam else None
    roofline = None
    if dominant:
        d = fam[dominant]
        ach = d["bytes"] / (d["ms"] / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": dominant, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": _traffic(wl, dominant, rows), "peak_source": peak_src,
                    "avg_launch_ms": d["ms"] / d["launches"],
                    "algorithmic_bytes_per_launch": d["bytes"] / d["launches"],
                    "share_of_step": (d["ms"] / args.steps) / ms_per_step,
                    "whole_step_gbs": algo * rows / (ms_per_step / 1e3) / 1e9,
                    "whole_step_frac": algo * rows / (ms_per_step / 1e3) / 1e9 / peak}

    # ---------------- hashbucket: roofline curve over the row count -----------------
    sweep = None
    if wl == "hashbucket" and args.sweep:
        sweep = []
        for r in [int(float(x)) for x in args.sweep.split(",") if x]:
            r = min(r, rows) // 64 * 64
            sub = cut(table.slice_rows(0, r), max(1, round(args.parts * r / rows)))
            ms, _, _, _ = timed(sub, max(3, args.steps), 3, False)
            gbs = algo * r / (ms / 1e3) / 1e9
            sweep.append({"rows_per_gpu": r, "ms_per_step": ms, "rows_per_s": r * world / (ms / 1e3),
                          "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak})
            del sub

    # ---------------- the other artefact policies beside the timed one ----------------
    artifact_legs = None
    if wl == "criteo" and world == 1 and not args.no_e2e:
        artifact_legs = {}
        for mode in ("lazy", "eager"):
            if mode == args.artifacts:
                continue
            try:
                os.environ["NVTB_ARTIFACTS"] = mode
                ms, _, _, _ = timed(frame, max(1, min(args.steps, 3)), 1, False)
                artifact_legs[mode] = {"ms_per_step": ms, "value": total_rows / (ms / 1e3), "unit": "rows/s"}
            except Exception as exc:          # noqa: BLE001 - reported, not fatal
                artifact_legs[mode] = {"error": repr(exc)[:200]}
            finally:
                os.environ["NVTB_ARTIFACTS"] = args.artifacts

    # ---------------- end to end from pinned host buffers ---------------------------
    e2e = None
    if not args.no_e2e:
        try:
            # host footprint: the pinned-memory allocator rounds every buffer up to a power of two, and
            # the 1-GPU box's cgroup holds 200 GiB — partitions of exactly 2^23 rows (32 / 64 MiB
            # buffers) and at most 2^27 rows per GPU keep a step at ~64 GB of pinned memory
            e_rows = args.e2e_rows or min(rows, 1 << 27)
            if not args.e2e_rows:
                # 481 B per row of the Criteo table are pinned (inputs + int64/float64 results); the same
                # bound is applied to the other workloads, whose rows are narrower
                local = int(os.environ.get("LOCAL_WORLD_SIZE", world))
                e_rows = e2e_rows_within_host_memory(e_rows, E2E_PINNED_BYTES_PER_ROW, local, _host_memory_budget())
                if world > 1:
                    agree = torch.tensor([e_rows], dtype=torch.int64, device=dev)
                    dist.all_reduce(agree, op=dist.ReduceOp.MIN)
                    e_rows = int(agree.item())
            e_parts = args.e2e_parts or max(1, (e_rows + (1 << 23) - 1) >> 23)
            src = table.slice_rows(0, e_rows) if e_rows <= rows else make_table(wl, e_rows, dev, rank, args.profile_rows)
            host = host_partitions(src, e_parts)
            del src
            table = None
            # the device-resident table and the allocator blocks cached by the timed region above
            # are not part of the e2e leg: it starts from host buffers and a clean device pool
            frame = None
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            if os.environ.get("NVTB_BENCH_DUMP"):
                free, tot = torch.cuda.mem_get_info()
                sys.stderr.write("[bench dump] before e2e: torch allocated %.1f GB, reserved %.1f GB, device free %.1f of %.1f GB\n"
                                 % (torch.cuda.memory_allocated() / 1e9, torch.cuda.memory_reserved() / 1e9, free / 1e9, tot / 1e9))
            out_host = None
            # W >= 3 warm-up steps here too: the first e2e step pins the result buffers (seconds),
            # the second still grows the device allocator's pools
            for _ in range(max(3, args.warmup)):
                h2d, d2h, out_host = run_step_e2e(nvt, wf, host, out_host, has_fit)
            sync_all()
            e_steps = max(1, min(args.steps, 3))
            t0 = time.perf_counter()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(e_steps):
                h2d, d2h, out_host = run_step_e2e(nvt, wf, host, out_host, has_fit)
            ev1.record()
            sync_all()
            e_ms = max(ev0.elapsed_time(ev1), (time.perf_counter() - t0) * 1e3)
            t = torch.tensor([e_ms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = float(t.item()) / e_steps
            e2e = {"value": e_rows * world / (e_ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": h2d * world,
                   "d2h_bytes_per_step": d2h * world, "ms_per_step": e_ms, "rows_per_step": e_rows * world,
                   "host_partitions_per_gpu": len(host), "warmup": max(3, args.warmup), "steps": e_steps,
                   "numa_node": numa,
                   # fit needs every partition before the first label exists, so H2D and D2H of one
                   # step cannot overlap: the bound is their SUM at the ~55 GB/s one PCIe 5 x16 sustains
                   "pcie_serial_bound_ms": (h2d + d2h) / 55e9 * 1e3 if has_fit else max(h2d, d2h) / 55e9 * 1e3}
            del host, out_host
        except Exception as exc:          # noqa: BLE001
            # a failed e2e leg must not cost the device-resident line on a single GPU; with several
            # ranks the others are inside collectives, so the error is re-raised there
            if world > 1:
                raise
            e2e = {"error": repr(exc)[:300]}

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_rows = args.cpu_rows or CPU_SAMPLE_ROWS[wl][0]
        v, sec, _, cpu_rows = cpu_reference(wl, cpu_rows, 1, args.profile_rows, budget_s=20.0)
        cpu_baseline = {"value": v, "unit": "rows/s", "cores": 1, "cpu_model": _cpu_model(), "kind": "port",
                        "sample": f"{cpu_rows} rows of the same synthetic table, "
                                  f"{'fit+transform' if has_fit else 'transform'}, {sec:.1f} s on 1 core "
                                  f"(host has {os.cpu_count()})"}

    line = {
        "metric": METRIC[wl], "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": {"criteo": "int32" if args.int32_outputs else "int64", "hashbucket": "u64", "movielens": "f64"}[wl],
        "data": "synthetic", "config": workload_config(args, world, rows),
        "roofline": roofline, "kernels": kernels, "e2e": e2e, "first_fit_ms": first_fit_ms,
        "parity_gate": gate, "artifact_policies": artifact_legs, "sweep": sweep,
        "cpu_baseline": cpu_baseline, "gpu_launches": launches, "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
