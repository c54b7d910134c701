"""Session-op benchmark: the Transformers4Rec preprocessing of reference tests/unit/test_tf4rec.py
(Groupby by session sorted by time, then ListSlice(-20, pad=True)) on one partition of 2.5e8
events, for two session-length distributions:

  poisson      lengths ~ 1 + Poisson(9): mean 10 events
  heavy_tail   1 % of the sessions hold half of the events (500 each), the rest ~ Poisson

Prints one JSON line: ms per step and events/s (CUDA events, after warm-up), the algorithmic bytes
of a step (inputs read once + outputs written once, the least any implementation moves) and the
share of 7.7 TB/s they imply, the GPU's name and power limit, parity with the CPU oracle on a
seeded sample of sessions, and the same step composed from torch ops (stable argsorts,
index_select, scatter_reduce) with its outputs asserted equal.  Needs a CUDA device; there is no
fallback.

    python tools/bench_sessions.py [--rows 250000000] [--steps 10] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

AGGS = {"item_id": ["list", "count"], "price": ["list", "mean"], "ts": ["first", "last"]}
MAX_LEN = 20
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def make_events(rows, kind, seed):
    """session_id, ts, item_id (int64), price (float32) on the device, sessions interleaved"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "poisson":
        lens = 1 + torch.poisson(torch.full((rows // 10 + 16,), 9.0, device="cuda"), generator=g).long()
    else:
        n_sessions = rows // 10
        heavy = max(1, n_sessions // 100)
        light = torch.poisson(torch.full((n_sessions - heavy,), 4.0, device="cuda"), generator=g).long() + 1
        lens = torch.cat([torch.full((heavy,), (rows // 2) // heavy, device="cuda", dtype=torch.long), light])
    sid = torch.repeat_interleave(torch.arange(lens.numel(), device="cuda"), lens)[:rows]
    if sid.numel() < rows:
        sid = torch.cat([sid, torch.arange(rows - sid.numel(), device="cuda") + lens.numel()])
    sid = sid[torch.randperm(rows, device="cuda", generator=g)] * 7919 + 10**9
    ts = torch.randint(1_600_000_000, 1_700_000_000, (rows,), device="cuda", generator=g)
    item = torch.randint(0, 1_000_000, (rows,), device="cuda", generator=g)
    price = torch.rand(rows, device="cuda", generator=g, dtype=torch.float32) * 100
    return {"session_id": sid, "ts": ts, "item_id": item, "price": price}


def build_workflow(nvt):
    ops = nvt.ops
    sessions = ["session_id", "item_id", "ts", "price"] >> ops.Groupby(
        groupby_cols=["session_id"], sort_cols=["ts"], aggs=AGGS, name_sep="-")
    seqs = sessions["item_id-list", "price-list"] >> ops.ListSlice(-MAX_LEN, pad=True)
    return nvt.Workflow(sessions["session_id", "item_id-count", "price-mean", "ts-first", "ts-last"] + seqs)


def torch_step(ev):
    """the same outputs from torch ops on the same device"""
    o1 = torch.argsort(ev["ts"], stable=True)
    perm = o1.index_select(0, torch.argsort(ev["session_id"].index_select(0, o1), stable=True))
    sid = ev["session_id"].index_select(0, perm)
    keys, counts = torch.unique_consecutive(sid, return_counts=True)
    group = torch.repeat_interleave(torch.arange(keys.numel(), device=sid.device), counts)
    ends = torch.cumsum(counts, 0)
    starts = ends - counts
    ts = ev["ts"].index_select(0, perm)
    psum = torch.zeros(keys.numel(), dtype=torch.float64, device=sid.device).scatter_reduce(
        0, group, ev["price"].index_select(0, perm).double(), "sum")
    take = torch.clamp(counts, max=MAX_LEN)
    j = torch.arange(MAX_LEN, device=sid.device)
    src = (ends - take).unsqueeze(1) + j
    valid = j < take.unsqueeze(1)
    src = torch.where(valid, src, torch.zeros_like(src))
    out = {"session_id": keys, "item_id-count": counts.int(), "price-mean": (psum / counts).float(),
           "ts-first": ts.index_select(0, starts), "ts-last": ts.index_select(0, ends - 1)}
    for c in ("item_id", "price"):
        v = ev[c].index_select(0, perm).index_select(0, src.reshape(-1)).reshape(src.shape)
        out[f"{c}-list"] = torch.where(valid, v, torch.zeros_like(v))
    return out


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        out = fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / steps, out


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def parity(out, ev, n_sample, seed):
    """engine output == oracle (oracle/sessions.py) on a seeded sample of sessions"""
    from oracle import sessions as osess
    rng = np.random.default_rng(seed)
    keys = out["session_id"].data.cpu().numpy()
    pick = np.sort(rng.choice(len(keys), min(n_sample, len(keys)), replace=False))
    pick_t = torch.from_numpy(keys[pick]).cuda()
    rows = torch.isin(ev["session_id"], pick_t).nonzero().squeeze(1)
    df = pd.DataFrame({c: t.index_select(0, rows).cpu().numpy() for c, t in ev.items()})
    exp = osess.groupby(df, ["session_id"], ["ts"], AGGS, name_sep="-")
    ok = np.array_equal(exp["session_id"].to_numpy(), keys[pick])
    for c in ("item_id-count", "ts-first", "ts-last"):
        ok &= np.array_equal(exp[c].to_numpy(), out[c].data.cpu().numpy()[pick])
    ok &= np.allclose(exp["price-mean"].to_numpy(), out["price-mean"].data.cpu().numpy()[pick], rtol=1e-6)
    for c in ("item_id-list", "price-list"):
        want = np.array(osess.list_slice(exp[c], -MAX_LEN, pad=True), dtype=np.float64)
        got = out[c].data.cpu().numpy().reshape(-1, MAX_LEN)[pick].astype(np.float64)
        ok &= np.array_equal(want, got)
    return bool(ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=250_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sample", type=int, default=10_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sessions.py needs a CUDA device (B200); there is no CPU path")
    import nvtabular as nvt
    from nvtabular_b200.column import Column, DeviceFrame
    name, power = gpu_identity()
    result = {"bench": "sessions", "rows": args.rows, "steps": args.steps, "warmup": args.warmup,
              "gpu": name, "power_limit": power, "workloads": {}}
    for i, kind in enumerate(("poisson", "heavy_tail")):
        ev = make_events(args.rows, kind, 1234 + i)
        frame = DeviceFrame({k: Column(v) for k, v in ev.items()})
        wf = build_workflow(nvt)
        ms, out = timed(lambda: wf.transform(frame), args.steps, args.warmup)
        n_groups = len(out)
        torch_ms, ref = timed(lambda: torch_step(ev), args.steps, args.warmup)
        same = all(torch.equal(out[c].data.view(-1), ref[c].view(-1))
                   for c in ("session_id", "item_id-count", "ts-first", "ts-last", "item_id-list", "price-list"))
        same &= bool(torch.allclose(out["price-mean"].data, ref["price-mean"], rtol=1e-6))
        assert same, f"{kind}: engine and torch composition disagree"
        nbytes = args.rows * 28 + n_groups * (8 + 4 + 4 + 8 + 8 + MAX_LEN * (8 + 4))
        result["workloads"][kind] = {
            "sessions": n_groups, "max_session": int(out["item_id-count"].data.max().item()),
            "ms_per_step": round(ms, 3), "events_per_s": args.rows / (ms / 1e3),
            "algorithmic_bytes": nbytes, "share_of_7.7TBps": nbytes / (ms / 1e3) / HBM_BYTES_PER_S,
            "torch_ms_per_step": round(torch_ms, 3), "speedup_vs_torch": round(torch_ms / ms, 3),
            "outputs_equal_torch": same, "parity": parity(out, ev, args.sample, 99 + i)}
        del frame, out, ref, ev
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
