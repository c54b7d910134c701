"""torchrun worker (NCCL, one rank per GPU) for tests/test_dist_gpu.py: every rank fits the
Criteo-shaped workflow on ITS shard; the fitted vocabularies / statistics must equal a
single-process fit over the concatenation of all shards, and the transform of the local
shard must equal the single-process transform of those rows."""
import os
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    import nvtabular_b200 as nvt
    from nvtabular_b200.column import Column, DeviceFrame
    from nvtabular_b200.synth import CAT_NAMES, CONT_NAMES, criteo_frame

    # C1 / C20 at ~2e6 keys with the sorted-accumulator threshold lowered: the key-range exchange
    # of packed pairs (dist.global_merge_sorted) runs next to the key-hash exchange of the small
    # columns; odd ranks hold a quarter of the rows, so their C1 / C20 start as hash tables and
    # are converted (nvtb_hashagg_to_sorted) when the ranks agree on the representation
    os.environ["NVTB_RUNS_MIN_KEYS"] = "300000"
    cats, conts = CAT_NAMES[:8] + ["C20"], CONT_NAMES[:4]
    shards = [criteo_frame((1 << 20) if r % 2 == 0 else (1 << 18), total_rows=40_000_000, device="cuda", rank=r)
              for r in range(world)]
    mine = shards[rank]

    def workflow(path):
        return nvt.Workflow((cats >> nvt.ops.Categorify(out_path=path, freq_threshold=2))
                            + (conts >> nvt.ops.FillMissing() >> nvt.ops.Normalize()))

    tmp = tempfile.TemporaryDirectory(prefix=f"nvtb_dist_rank{rank}_")

    # distributed fit on the local shard
    wf = workflow(os.path.join(tmp.name, "dist"))
    wf.fit(nvt.Dataset(mine))
    out = next(iter(wf.transform(nvt.Dataset(mine)).partitions()))

    # reference: the same engine, single process, all shards as partitions (no collectives)
    os.environ["NVTB_DISABLE_DIST"] = "1"
    ref = workflow(os.path.join(tmp.name, "single"))
    ref.fit(nvt.Dataset(shards))
    ref_out = ref.transform(mine)
    os.environ.pop("NVTB_DISABLE_DIST")

    cat_op = [n.op for n in wf.output_node.topo_order() if type(n.op).__name__ == "Categorify"][0]
    modes = {c: cat_op._aggs[c].mode for c in cats}
    # (with the threshold this low a blind first batch sends the small columns down the same path:
    # counts up to 2^20 then exercise the multi-pass count ordering of the owners' shards)
    assert modes["C1"] == 1 and modes["C20"] == 1, modes
    ref_op = [n.op for n in ref.output_node.topo_order() if type(n.op).__name__ == "Categorify"][0]
    for c in cats:
        k1, s1 = cat_op.categories.fitted[c].vocab.export()
        k2, s2 = ref_op.categories.fitted[c].vocab.export()
        assert torch.equal(k1, k2) and torch.equal(s1, s2), f"vocab mismatch for {c} on rank {rank}"
        v1, v2 = cat_op.categories.fitted[c].vocab, ref_op.categories.fitted[c].vocab
        assert (v1.null_size, v1.oov_size, v1.unique_size) == (v2.null_size, v2.oov_size, v2.unique_size)
        assert torch.equal(out[c].data, ref_out[c].data), f"labels differ for {c} on rank {rank}"
    n1 = [n.op for n in wf.output_node.topo_order() if type(n.op).__name__ == "Normalize"][0]
    n2 = [n.op for n in ref.output_node.topo_order() if type(n.op).__name__ == "Normalize"][0]
    for c in conts:
        assert abs(n1.means[c] - n2.means[c]) <= 1e-12 * max(1.0, abs(n2.means[c]))
        assert abs(n1.stds[c] - n2.stds[c]) <= 1e-12 * max(1.0, abs(n2.stds[c]))
    dist.barrier()
    if rank == 0:
        print(f"DIST_OK world={world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
