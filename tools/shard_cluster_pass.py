#!/usr/bin/env python
"""tools/shard_cluster_pass.py -- the sample-sharded cluster pass (shard.cluster_pass_sharded) on bench.py's workloads, one GPU per rank.

  torchrun --nproc-per-node N tools/shard_cluster_pass.py --config K [--scale S] [--no-check]

Rank r generates only the samples k with k % N == r of the configs[K] job (Synth.sample(k, ...), packed with sample_ids=[k ...]),
cuts them by the batching rule and runs the pass twice (warm-up, then timed).  Per rank it reports the bundles, hits and bytes sent
and received, the exchange time (host clock around synchronised work), every phase and the largest rank time over the mean; as the
ceiling of the exchange, a plain NCCL all-to-all of the same byte counts between torch tensors, timed the same way.  Rank 0 then runs
the whole job through the single-GPU clusters.cluster_pass and reports the bundles whose digests (bench.view_digests) differ, the
clusters whose support rows differ and whether the clusters are identical.  Prints one JSON line on rank 0; progress goes to stderr."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench                                                   # noqa: E402
import cluster_pass as single                                  # noqa: E402  (tools/cluster_pass.py: card(), same_rows())
from aletsch_b200 import clusters as CL                        # noqa: E402
from aletsch_b200 import gpu as G                              # noqa: E402
from aletsch_b200 import hostlib as H                          # noqa: E402
from aletsch_b200 import shard                                 # noqa: E402


def generate(cfg, samples):
    """records of the given samples of the configs[K] job (bench.build_workload's generator: rank 0's chromosomes)"""
    kw = {"expressed_fraction": cfg["expressed_fraction"]} if "expressed_fraction" in cfg else {}
    sc = H.default_config(cfg["mode_id"], chrom_len=cfg["chrom_len"], n_chrom=cfg["n_chrom"], seed=cfg["seed"], **kw)
    syn = H.Synth(sc)
    return [syn.sample(k, cfg["per_sample"], threads=8) for k in samples]


def run_pass(ctx, parts, srcs, keys, gp, times=None):
    for s in srcs:
        s.reset()
    return shard.cluster_pass_sharded(ctx, parts, srcs, keys, gp, support=True, times=times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=1)
    ap.add_argument("--scale", type=float, default=None)
    ap.add_argument("--no-check", action="store_true", help="skip the single-GPU run of the whole job on rank 0")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    card = single.card() if rank == 0 else None
    cfg = bench.config_of(args)
    mine = [k for k in range(cfg["samples"]) if k % world == rank]
    t0 = time.time()
    batch = H.pack(generate(cfg, mine), H.default_packer_params(cfg["library_type"]), sample_ids=mine)
    bench.log("[shard_cluster_pass] rank %d: %d samples, %d bundles, %d hits in %.1fs" % (rank, len(mine), batch.n_bundles, batch.n_hits,
                                                                                      time.time() - t0))
    gp = G.default_params(library_type=cfg["library_type"], min_junction_support=cfg.get("min_junction_support", 1), **cfg["group"])
    ctx = G.Context(local)
    parts = CL.device_batches(batch) if batch.n_bundles else []
    srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
    keys = shard.bundle_keys(batch)

    run_pass(ctx, parts, srcs, keys, gp).free()
    dist.barrier()
    times = {}
    t0 = time.perf_counter()
    res = run_pass(ctx, parts, srcs, keys, gp, times)
    total = time.perf_counter() - t0
    ex = res.exchange
    digests = {}
    for b, o in zip(res.batches, res.origin):
        d = bench.view_digests(b.results(G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS), len(o))
        digests.update(zip(o[:, 1].tolist(), map(tuple, d.tolist())))
    clusters = [[int(o[m, 1]) for m in c] for o, cl in zip(res.origin, res.clusters) for c in cl]
    rows = [d for s in res.support for d in s]
    res.free()

    # the ceiling: one NCCL all-to-all of the same byte counts between torch tensors
    dev = torch.device("cuda", local)
    src = torch.zeros(max(sum(ex["bytes_to"]), 1), dtype=torch.int8, device=dev)
    dst = torch.empty(max(sum(ex["bytes_from"]), 1), dtype=torch.int8, device=dev)
    a2a = []
    for it in range(3):
        dist.barrier()
        torch.cuda.synchronize()
        ta = time.perf_counter()
        dist.all_to_all_single(dst[:sum(ex["bytes_from"])], src[:sum(ex["bytes_to"])], output_split_sizes=ex["bytes_from"],
                               input_split_sizes=ex["bytes_to"])
        torch.cuda.synchronize()
        a2a.append(time.perf_counter() - ta)
    del src, dst
    me = {"rank": rank, "samples": len(mine), "bundles": batch.n_bundles, "hits": batch.n_hits, "source_batches": len(parts),
          "exchange": {k: v for k, v in ex.items()}, "exchange_s": round(times["exchange"], 4),
          "exchange_gbs": round((ex["bytes_sent"] + ex["bytes_received"]) / times["exchange"] / 1e9, 2) if times["exchange"] > 0 else None,
          "all_to_all_s": round(min(a2a), 4),
          "all_to_all_gbs": round((ex["bytes_sent"] + ex["bytes_received"]) / min(a2a) / 1e9, 2) if min(a2a) > 0 else None,
          "owned_hits": int(res.load[rank]) if hasattr(res, "load") else 0, "output_batches": len(res.origin),
          "seconds": {k: (round(v, 4) if not isinstance(v, list) else [round(x, 4) for x in v]) for k, v in times.items()},
          "seconds_total": round(total, 4)}
    every = [None] * world
    dist.all_gather_object(every, (me, digests, clusters, rows))
    for s in srcs:
        s.free()
    if rank == 0:
        tot = [e[0]["seconds_total"] for e in every]
        out = {"config": args.config, "card": card, "ranks": world, "per_rank": [e[0] for e in every],
               "largest_rank_time_over_mean": round(max(tot) / (sum(tot) / len(tot)), 3),
               "timing": "host clock around synchronised work, second pass after a warm-up"}
        if not args.no_check:
            bench.log("[shard_cluster_pass] single-GPU run of the whole job on rank 0")
            whole = H.pack(generate(cfg, range(cfg["samples"])), H.default_packer_params(cfg["library_type"]))
            wparts = CL.device_batches(whole)
            wsrc = [ctx.upload(p.view(), keepalive=p) for p in wparts]
            want = CL.cluster_pass(ctx, wparts, wsrc, gp, support=True)
            for s in wsrc:
                s.free()
            wkeys = shard.bundle_keys(whole)
            got_dig = {k: v for e in every for k, v in e[1].items()}
            bad = len(wkeys) - len(got_dig)
            for b, o in zip(want.batches, want.origin):
                d = bench.view_digests(b.results(G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS), len(o))
                bad += sum(got_dig.get(int(k)) != tuple(x) for k, x in zip(wkeys[o[:, 2]], d.tolist()))
            want_clusters = [[int(wkeys[o[m, 2]]) for m in c] for o, cl in zip(want.origin, want.clusters) for c in cl]
            want_rows = {tuple(c): r for c, r in zip(want_clusters, (d for s in want.support for d in s))}
            got = {tuple(c): r for e in every for c, r in zip(e[2], e[3])}
            out["check"] = {"bundles": len(wkeys), "clusters": len(want_clusters), "mismatching_bundle_digests": int(bad),
                            "clusters_identical": sorted(want_rows) == sorted(got),
                            "mismatching_support_rows": sum(c not in got or not single.same_rows(r, got[c]) for c, r in want_rows.items())}
            want.free()
        print(json.dumps(out))
    ctx.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
