"""Multi-GPU per-cell exchange check, launched one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29541 tests/multigpu_cells_check.py [n_reads]

Every rank pushes its contiguous run of a seeded set of files (one push per file, last read dropped, rank-major
order keys) on its own B200, with its OWN cell ids; the ranks merge their cell names into global ids and run
multi_gpu.distributed_finalize_cells.  Every rank's slice must be exactly its EC-id range of what the C oracle
computes for all files in order.  N = 1 runs the whole orchestration with a single rank.  One OK line per case."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def check(label, out, want, dev):
    a, b = out["id_base"], out["id_base"] + out["n_ec_local"]
    ip, ix, dt = want["a_indptr"], want["a_indices"], want["a_data"]
    n_ip, n_ix, n_dt = want["n_indptr"], want["n_indices"].astype(np.int64), want["n_data"]
    S = len(n_ip) - 1
    ok = (out["n_ec"] == len(ip) - 1 and out["n_samples"] == S
          and np.array_equal(out["cell_order"].cpu().numpy(), want["cell_order"])
          and np.array_equal(out["n_indptr"].cpu().numpy(), n_ip)
          and np.array_equal(out["a_indptr"].cpu().numpy(), ip[a:b + 1] - ip[a])
          and np.array_equal(out["a_indices"].cpu().numpy(), ix[ip[a]:ip[b]])
          and np.array_equal(out["a_data"].cpu().numpy(), dt[ip[a]:ip[b]]))
    if ok:   # this rank's N entries, column by column, at n_indptr[c] + n_col_offset[c]
        counts, offset = out["n_col_counts"].cpu().numpy(), out["n_col_offset"].cpu().numpy()
        idx, dat = out["n_indices"].cpu().numpy().astype(np.int64) + a, out["n_data"].cpu().numpy()
        at = 0
        for c in range(S):
            s = n_ip[c] + offset[c]
            k = counts[c]
            rows = n_ix[n_ip[c]:n_ip[c + 1]]
            ok = ok and k == ((rows >= a) & (rows < b)).sum() and np.array_equal(idx[at:at + k], n_ix[s:s + k]) \
                and np.array_equal(dat[at:at + k], n_dt[s:s + k])
            at += k
        ok = ok and at == len(idx)
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if dist.get_rank() == 0:
        print("multigpu_cells_check world=%d %s ECs=%d cells=%d: %s" % (dist.get_world_size(), label, len(ip) - 1, S,
                                                                        "OK" if flag.item() else "MISMATCH"), flush=True)
    if not flag.item():
        dist.destroy_process_group()
        sys.exit(1)


def main():
    n_reads = int(sys.argv[1]) if len(sys.argv) > 1 else 400000
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import datetime
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    from alntools_b200 import multi_gpu, synth
    from alntools_b200._native import EcBuilder
    from alntools_b200.bam_utils_multisample import RANK_STRIDE, merge_cell_names, partition_files
    from oracle import c_oracle

    # (seed, files, cells, min count); the second case has fewer files than 4 ranks would need
    for seed, n_files, n_cells, min_count, passes in ((21, 2 * world + 1, 3000, 20, 2), (22, max(1, world - 1), 500, 0, 1)):
        cols = synth.make_columns(n_reads, 20000, 2, seed=seed, mode="diploid", n_cells=n_cells, dup_rate=0.01)
        cuts = multi_gpu.shard_bounds(cols["read_group"], n_files)
        names = ["cell%05d" % c for c in range(n_cells)]
        files = [{k: np.ascontiguousarray(cols[k][cuts[i]:cuts[i + 1]]) for k in ("read_group", "target_idx", "hap_idx", "cell_idx")}
                 for i in range(n_files)]
        want = c_oracle.ec_from_columns_cells([(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], True)
                                               for f in files], min_count)
        fc = partition_files([len(f["read_group"]) for f in files], world)
        mine = files[fc[rank]:fc[rank + 1]]
        # this rank's own cell ids: first appearance over its files (as its CellDictionary gives them)
        seen = {}
        for f in mine:
            for g in f["cell_idx"].tolist():
                seen.setdefault(g, len(seen))
        lut = np.zeros(n_cells, dtype=np.int32)
        for g, l in seen.items():
            lut[g] = l
        local_b = EcBuilder(20000, 2, with_cells=True, device=local, result_on_device=1)
        owner_b = EcBuilder(20000, 2, device=local)
        lists = [None] * world
        dist.all_gather_object(lists, [names[g] for g in seen])
        gnames, maps = merge_cell_names(lists)
        cell_map = torch.from_numpy(maps[rank]).to(dev) if len(maps[rank]) else None
        for _ in range(passes):   # contexts (and arenas) are kept from pass to pass, as in a long-running job
            local_b.reset()
            owner_b.reset()
            base = rank * RANK_STRIDE
            for f in mine:
                local_b.push(f["read_group"], f["target_idx"], f["hap_idx"], np.ascontiguousarray(lut[f["cell_idx"]]),
                             order_base=base, drop_last_group=True)
                base += len(f["read_group"])
            out = multi_gpu.distributed_finalize_cells(local_b, lambda: owner_b, dev, min_count, cell_map, len(gnames))
        out = dict(out, cell_order=torch.tensor([int(gnames[g][4:]) for g in out["cell_order"].tolist()]))
        check("files=%d cells=%d min_count=%d" % (n_files, n_cells, min_count), out, want, dev)
        local_b.close()
        owner_b.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
