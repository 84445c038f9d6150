"""Multi-GPU parity check, launched one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29533 tests/multigpu_check.py [n_reads]

Every rank builds its contiguous shard of a seeded synthetic workload on its own B200, the ranks
exchange their ECs over peer memory (alntools_b200/multi_gpu.py) and every rank must end up with its
EC-id range of exactly the matrices the C oracle computes for the whole, unsharded input.  N = 1 runs
the whole orchestration with a single rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def check_slice(label, sl, oracle, dev):
    """This rank's slice must be rows [id_base, id_base + n_ec_local) of the oracle's matrices; one line per case."""
    indptr, indices, data, counts = oracle[:4]
    a, b = sl["id_base"], sl["id_base"] + sl["n_ec_local"]
    ok = (sl["n_ec"] == len(counts)
          and np.array_equal(sl["a_indptr"].cpu().numpy(), indptr[a:b + 1] - indptr[a])
          and np.array_equal(sl["a_indices"].cpu().numpy(), indices[indptr[a]:indptr[b]])
          and np.array_equal(sl["a_data"].cpu().numpy(), data[indptr[a]:indptr[b]])
          and np.array_equal(sl["n_data"].cpu().numpy(), counts[a:b]))
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if dist.get_rank() == 0:
        print("multigpu_check world=%d %s ECs=%d: %s" % (dist.get_world_size(), label, len(counts),
                                                           "OK" if flag.item() else "MISMATCH"), flush=True)
    if not flag.item():
        dist.destroy_process_group()
        sys.exit(1)


def main():
    n_reads = int(sys.argv[1]) if len(sys.argv) > 1 else 400000
    passes = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import datetime
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    from alntools_b200 import multi_gpu, synth
    from alntools_b200._native import EcBuilder
    from oracle import c_oracle

    for seed, mode, n_targets, n_haps in ((11, "diploid", 20000, 2), (12, "heavy", 3000, 8)):
        reads = n_reads if mode == "diploid" else n_reads // 20
        cols = synth.make_columns(reads, n_targets, n_haps, seed=seed, mode=mode, dup_rate=0.01)
        rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
        cuts = multi_gpu.shard_bounds(rg, world)
        a, b = cuts[rank], cuts[rank + 1]
        local_b = EcBuilder(n_targets, n_haps, alignments_hint=b - a, device=local)
        owner_b = EcBuilder(n_targets, n_haps, alignments_hint=b - a, device=local)
        for _ in range(passes):   # contexts are reused from pass to pass, as a long-running job would
            local_b.reset()
            owner_b.reset()
            local_b.push(np.ascontiguousarray(rg[a:b]), np.ascontiguousarray(tg[a:b]),
                         np.ascontiguousarray(hp[a:b]), order_base=a)
            sl = multi_gpu.distributed_finalize(local_b, lambda: owner_b, dev, result_on="slices")
        check_slice("mode=%s reads=%d alignments=%d" % (mode, reads, len(rg)), sl,
                    c_oracle.ec_from_columns(rg, tg, hp), dev)
        local_b.close()
        owner_b.close()

    # the bench's shape: every rank has its OWN seeded shard, columns resident on the device
    n_targets, n_haps = 20000, 2
    shards = [synth.make_columns(n_reads // 2, n_targets, n_haps, seed=100 + r, mode="diploid") for r in range(world)]
    sizes = [len(s["read_group"]) for s in shards]
    base = sum(sizes[:rank])
    mine = {k: torch.from_numpy(shards[rank][k]).to(dev) for k in ("read_group", "target_idx", "hap_idx")}
    local_b = EcBuilder(n_targets, n_haps, alignments_hint=sizes[rank], device=local, result_on_device=1)
    owner_b = EcBuilder(n_targets, n_haps, alignments_hint=sizes[rank], device=local)
    for _ in range(passes + 1):
        local_b.reset()
        owner_b.reset()
        local_b.push(mine["read_group"], mine["target_idx"], mine["hap_idx"], order_base=base)
        sl = multi_gpu.distributed_finalize(local_b, lambda: owner_b, dev, result_on="slices")
    rg = np.concatenate([s["read_group"] + 10 ** 8 * r for r, s in enumerate(shards)])   # reads stay distinct
    tg = np.concatenate([s["target_idx"] for s in shards])
    hp = np.concatenate([s["hap_idx"] for s in shards])
    check_slice("own-shards device-resident reuse: alignments=%d" % len(rg), sl,
                c_oracle.ec_from_columns(rg.astype(np.int32), tg, hp), dev)
    local_b.close()
    owner_b.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
