"""Command line: BAM files in, per-bundle evidence / splice graphs / bridged fragments / phasing paths on the GPU.

    python -m aletsch_b200.run [--library-type unstranded|first|second|auto] [--device 0] [--clusters] a.bam [b.bam ...]
    torchrun --nproc-per-node 2 -m aletsch_b200.run --clusters a.bam b.bam c.bam

One sample per BAM.  The files are decoded on the host (host/bamio.cc), cut into bundles by the packer (the record loop of
meta/generator.cc:77-201), and cut by position into device batches (clusters.device_batches, include/aletsch_gpu.h, BATCHING
RULE).  Without --clusters every device batch goes through bundle::bridge on its own.  With --clusters the bundles are clustered
across samples (bundle_group::resolve per 1 Mb region and strand), regrouped on the device cluster by cluster, bridged, and every
cluster is re-bridged against its combined splice graph (assembler::bridge): shard.cluster_pass_sharded.

Under torchrun (WORLD_SIZE > 1, one process per GPU, NCCL) the samples are sharded: rank r decodes the files with index
i % world == r, and with --clusters every cluster's bundles are moved to one GPU for the cluster pass.  One process is the same
run with one rank.  Rank 0 prints one JSON line with the totals over all ranks, with the same keys in every mode; the results
themselves are available through the fetch calls of aletsch_b200.gpu.Batch (this tool is a usage example, not a replacement for
the assembler).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

from .clusters import device_batches
from . import gpu as G
from . import hostlib as H
from .shard import bundle_keys, cluster_pass_sharded

REGION = 1_000_000


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m aletsch_b200.run")
    ap.add_argument("bams", nargs="+")
    ap.add_argument("--library-type", default="first", choices=["unstranded", "first", "second", "auto"],
                    help="auto: previewer::infer_library_type over the first file's records")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--clusters", action="store_true", help="cross-sample clustering (-c 20 -s 0.2 style) + group-level re-bridge")
    ap.add_argument("--max-group-size", type=int, default=200)
    ap.add_argument("--min-grouping-similarity", type=float, default=0.10)
    ap.add_argument("--whole-file", action="store_true",
                    help="one record loop per file instead of the reference's region table (sample_profile::set_batch_boundaries), "
                         "which drops every region's first hit and the last region of the last chromosome")
    args = ap.parse_args(argv)
    lt = {"unstranded": H.UNSTRANDED, "first": H.FR_FIRST, "second": H.FR_SECOND, "auto": None}[args.library_type]
    if int(os.environ.get("WORLD_SIZE", "1")) == 1:
        return _run(args, lt, 0, 1, args.device)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        return _run(args, lt, dist.get_rank(), dist.get_world_size(), local)
    finally:
        dist.destroy_process_group()


def _run(args, lt, rank, world, device):
    """rank `rank` of `world`: its files (index i % world == rank) through the device; collectives only when world > 1"""
    t0 = time.time()
    mine = [i for i in range(len(args.bams)) if i % world == rank]
    recs, chrom_len = [], None
    for i in mine:
        r, cl = H.read_bam(args.bams[i])
        if chrom_len is not None and not np.array_equal(cl, chrom_len):
            raise SystemExit("%s: reference dictionary differs from the first file's" % args.bams[i])
        chrom_len = cl
        recs.append(r)
        print("%s%s: %d records" % ("rank %d: " % rank if world > 1 else "", args.bams[i], r["n"]), file=sys.stderr)
    if world > 1:
        dicts = [None] * world
        dist.all_gather_object(dicts, None if chrom_len is None else [int(x) for x in chrom_len])
        chrom_len = np.array(dicts[0], np.int32)     # rank 0 holds file 0
        for r, d in enumerate(dicts):
            if d is not None and not np.array_equal(d, chrom_len):      # file r is the first file of rank r
                raise SystemExit("%s: reference dictionary differs from the first file's" % args.bams[r])
    if lt is None:
        got = [None]
        if rank == 0:
            pv = H.infer_library_type(recs[0], H.default_packer_params(H.UNSTRANDED))
            got[0] = pv["library_type"]
            print("inferred library type %d from %s: %s" % (got[0], args.bams[0], pv), file=sys.stderr)
        if world > 1:
            dist.broadcast_object_list(got, src=0)
        lt = got[0]
    batch = H.pack(recs, H.default_packer_params(lt), sample_ids=mine, chrom_len=None if args.whole_file else chrom_len,
                   region_length=REGION)
    t1 = time.time()
    gp = G.default_params(library_type=lt, max_group_size=args.max_group_size, min_grouping_similarity=args.min_grouping_similarity)
    ctx = G.Context(device)
    parts = device_batches(batch) if batch.n_bundles else []
    out = {"samples": len(recs), "bundles": batch.n_bundles, "decode_pack_s": t1 - t0, "device_batches": len(parts)}
    if args.clusters:
        srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
        res = cluster_pass_sharded(ctx, parts, srcs, bundle_keys(batch), gp)
        for s in srcs:
            s.free()
        out["region_groups"] = res.n_groups
        out["clusters_of_bundles"] = sum(len(c) for c in res.clusters)
        bts = res.batches
    else:
        def bridged(p):
            bt = ctx.upload(p.view(), keepalive=p)
            bt.bridge_all(gp)
            return bt
        bts = (bridged(p) for p in parts)
    out.update(dict.fromkeys((n for n, _ in G.Counts._fields_), 0))
    out["distinct_phases"] = 0
    for bt in bts:
        bt.graph(gp)
        out["distinct_phases"] += int(sum(len(p["phase_cnt"]) for p in bt.phase_set()))
        for n, v in bt.counts().items():
            out[n] += v
        bt.free()
    out["device_s"] = time.time() - t1
    ctx.close()
    if world > 1:
        every = [None] * world
        dist.all_gather_object(every, out)
        # seconds: the slowest rank; region_groups is a count of the whole job, the same on every rank
        out = {n: max(o[n] for o in every) if n.endswith("_s") or n == "region_groups" else sum(o[n] for o in every) for n in out}
    out["decode_pack_s"], out["device_s"] = round(out["decode_pack_s"], 3), round(out["device_s"], 3)
    out["ranks"] = world
    if rank == 0:
        print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
