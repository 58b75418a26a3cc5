"""One rank of the sample-sharded cluster pass with phases=True (tests/test_group_phase_set.py), spawned over gloo on the
kernel-logic build: every rank ingests its own samples (sample % world == rank), runs shard.cluster_pass_sharded and compares the
combined phase set of every cluster it owns with the whole job run as one device batch in this process.  Rank 0 checks that the
clusters of all ranks together are the single-batch clusters."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def run(lib_path=None, mode=None, samples=4, templates=8000, max_batch_hits=None):
    import torch.distributed as dist
    import parity
    import test_group_phase_set as T
    from aletsch_b200 import clusters as CL, gpu as G, hostlib as H, shard
    rank, world = dist.get_rank(), dist.get_world_size()
    mode = H.SYNTH_PAIRED if mode is None else mode
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    sample = batch.a["bundle_sample"].astype(np.int64)
    keys_all = (sample << 32) | np.arange(batch.n_bundles, dtype=np.int64)
    mine = np.nonzero(sample % world == rank)[0]
    sub = batch.select([int(k) for k in mine])
    parts = sub.split(2) if sub.n_bundles else []
    ctx = G.Context(0, lib_path=lib_path)
    srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
    if max_batch_hits:
        CL.MAX_BATCH_HITS = max_batch_hits
    res = shard.cluster_pass_sharded(ctx, parts, srcs, keys_all[mine], gp, phases=True)
    for s in srcs:
        s.free()
    whole, multi, _, px_want = T.single_batch_phases(ctx, batch, gp)
    index = {tuple(c): i for i, c in enumerate(multi)}
    bad, got, spanning = [], [], 0
    for o, cl, px in zip(res.origin, res.clusters, res.phases):
        job = o[:, 1] & 0xffffffff
        assert len(px) == len(cl)
        for c, d in zip(cl, px):
            members = tuple(int(job[m]) for m in c)
            got.append(list(members))
            spanning += len(set(o[c, 0].tolist())) > 1
            gi = index.get(members)
            if gi is None or not T.same(px_want[gi], d):
                bad.append("rank %d: cluster %s" % (rank, members))
    summary = {"rank": rank, "clusters": got, "spanning": spanning, "bad": bad[:20], "n_bad": len(bad)}
    res.free()
    whole.free()
    ctx.close()
    gathered = [None] * world
    dist.all_gather_object(gathered, summary)
    result = {"rank": rank, "clusters": len(multi), "spanning": sum(g["spanning"] for g in gathered)}
    if rank == 0:
        n_bad = sum(g["n_bad"] for g in gathered)
        assert n_bad == 0, "%d mismatches, first: %s" % (n_bad, [b for g in gathered for b in g["bad"]][:5])
        assert sorted(c for g in gathered for c in g["clusters"]) == sorted(multi), "the clusters of all ranks are the single-batch ones"
    dist.barrier()
    return result
