"""One rank of the sample-sharded cluster pass (tests/test_shard_cluster_pass.py): launched by torchrun (NCCL, one GPU per rank) or
spawned over gloo on the kernel-logic build.  Every rank ingests its own samples (sample % world == rank), runs
shard.cluster_pass_sharded, and compares what it owns with the whole job run as one device batch
(test_cluster_pass.single_batch_run): per bundle every view of agpu_batch_results(ALL) and bundle_counts, per cluster the combined
bundle and the support rows.  Rank 0 then checks that every bundle is in exactly one rank's output and that the clusters of all ranks
are the single-batch clusters, in order."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def run(backend, lib_path=None, mode=None, samples=4, templates=8000, max_batch_hits=None, out=None):
    import torch
    import torch.distributed as dist
    import parity
    import test_cluster_pass as T
    from aletsch_b200 import clusters as CL, gpu as G, hostlib as H, shard
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank)) if backend == "nccl" else 0
    if backend == "nccl":
        torch.cuda.set_device(local)
    mode = H.SYNTH_PAIRED if mode is None else mode
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    sample = batch.a["bundle_sample"].astype(np.int64)
    keys_all = (sample << 32) | np.arange(batch.n_bundles, dtype=np.int64)
    mine = np.nonzero(sample % world == rank)[0]
    sub = batch.select([int(k) for k in mine])
    parts = sub.split(2) if sub.n_bundles else []
    ctx = G.Context(local, lib_path=lib_path)
    srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
    if max_batch_hits:
        CL.MAX_BATCH_HITS = max_batch_hits          # several output batches per rank
    times = {}
    res = shard.cluster_pass_sharded(ctx, parts, srcs, keys_all[mine], gp, support=True, times=times)
    for s in srcs:
        s.free()
    # the oracle: the whole job as one device batch on this rank's device
    whole, multi, cb_want, sup_want = T.single_batch_run(ctx, batch, gp)
    per_bundle_want = whole.bundle_counts()
    cluster_index = {tuple(c): i for i, c in enumerate(multi)}
    hit_off = batch.a["bundle_hit_off"]
    nh = np.diff(hit_off)
    bad, got_clusters, owned, spanning = [], [], [], 0
    for i, (bt, o, cl) in enumerate(zip(res.batches, res.origin, res.clusters)):
        job = o[:, 1] & 0xffffffff
        assert np.array_equal(o[:, 1], keys_all[job])
        local_rows = o[:, 0] == rank
        assert np.all((o[:, 2] >= 0) == local_rows) and np.all((o[:, 3] >= 0) == local_rows)
        base = np.concatenate([[0], np.cumsum([p.n_bundles for p in parts])]).astype(np.int64)
        assert np.array_equal(mine[base[o[local_rows, 2]] + o[local_rows, 3]], job[local_rows]), "origin rows of local bundles"
        owned += job.tolist()
        loc_off = np.concatenate([[0], np.cumsum(nh[job])])
        bad += T.diff_arrays(T.all_results(whole, batch.n_bundles, hit_off, job), T.all_results(bt, len(o), loc_off), "rank %d batch %d" % (rank, i))
        if not np.array_equal(bt.bundle_counts(), per_bundle_want[job]):
            bad.append("rank %d batch %d: bundle_counts differ" % (rank, i))
        if not cl:
            continue
        cb = bt.fetch_group()
        for k, c in enumerate(cl):
            members = tuple(int(job[m]) for m in c)
            got_clusters.append(list(members))
            spanning += len(set(o[c, 0].tolist())) > 1
            gi = cluster_index.get(members)
            if gi is None:
                bad.append("rank %d: cluster %s is not a single-batch cluster" % (rank, members))
                continue
            bad += T.diff_arrays(cb_want[gi], cb[k], "cluster %d combined bundle" % gi)
            w, g = sup_want[gi], res.support[i][k]
            if sorted(w) != sorted(g):
                bad.append("cluster %d: support row names differ" % gi)
                continue
            for name in sorted(w):
                a, b = np.asarray(w[name]), np.asarray(g[name])
                (parity.cmp_f64 if a.dtype == np.float64 else parity.cmp_int)(name, a, b, "cluster %d support" % gi, bad)
    mine_summary = {"rank": rank, "owned": owned, "clusters": got_clusters, "spanning": spanning, "bad": bad[:20], "n_bad": len(bad),
                    "exchange": res.exchange, "n_clusters": res.n_clusters, "batches": len(res.batches), "times": sorted(times)}
    res.free()
    whole.free()
    ctx.close()
    gathered = [None] * world
    dist.all_gather_object(gathered, mine_summary)
    result = {"rank": rank, "world": world, "backend": backend, "ranks": gathered}
    if rank == 0:
        n_bad = sum(g["n_bad"] for g in gathered)
        assert n_bad == 0, "%d mismatches, first: %s" % (n_bad, [b for g in gathered for b in g["bad"]][:5])
        owned = sorted(k for g in gathered for k in g["owned"])
        assert owned == list(range(batch.n_bundles)), "every bundle in exactly one rank's output"
        assert sorted(c for g in gathered for c in g["clusters"]) == sorted(multi), "the clusters of all ranks are the single-batch ones"
        for g in gathered:
            pos = [cluster_index[tuple(c)] for c in g["clusters"]]
            assert pos == sorted(pos), "rank %d lays its clusters out in the single-batch order" % g["rank"]
        assert all(g["n_clusters"] == gathered[0]["n_clusters"] for g in gathered)
        result.update({"bundles": int(batch.n_bundles), "clusters": len(multi), "spanning": sum(g["spanning"] for g in gathered),
                       "bytes_sent": sum(g["exchange"]["bytes_sent"] for g in gathered)})
    dist.barrier()
    if out and rank == 0:
        json.dump(result, open(out, "w"))
    return result


if __name__ == "__main__":
    import torch
    import torch.distributed as dist
    backend = sys.argv[1] if len(sys.argv) > 1 else "nccl"
    out = sys.argv[2] if len(sys.argv) > 2 else None
    samples, templates = (int(sys.argv[3]), int(sys.argv[4])) if len(sys.argv) > 4 else (8, 40000)
    if backend == "nccl":
        dev = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo")
    r = run(backend, samples=samples, templates=templates, max_batch_hits=None, out=out)
    if dist.get_rank() == 0:
        print("shard_cluster_worker ok: %s" % json.dumps({k: v for k, v in r.items() if k != "ranks"}))
    dist.destroy_process_group()
