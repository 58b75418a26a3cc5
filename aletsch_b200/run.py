"""Command line: BAM files in, per-bundle evidence / splice graphs / bridged fragments / phasing paths on the GPU.

    python -m aletsch_b200.run [--library-type unstranded|first|second] [--device 0] [--clusters] a.bam [b.bam ...]

One sample per BAM.  The files are decoded on the host (host/bamio.cc), cut into bundles by the packer (the record loop of
meta/generator.cc:77-201), and the whole batch goes through bundle::bridge on the device; with --clusters the bundles are also
clustered across samples (bundle_group::resolve per 1 Mb region and strand) and every cluster is re-bridged against its combined
splice graph (assembler::bridge).  A job larger than one device batch (include/aletsch_gpu.h, BATCHING RULE) is cut by
position (clusters.device_batches); with --clusters its bundles are then regrouped on the device by cluster (clusters.cluster_pass).
Prints one summary line per sample and the totals; the results themselves are available
through the fetch calls of aletsch_b200.gpu.Batch (this tool is a usage example, not a replacement for the assembler).

Under torchrun (WORLD_SIZE > 1, one process per GPU, NCCL) the samples are sharded: rank r decodes the files with index
i % world == r, and with --clusters every cluster's bundles are moved to one GPU for the cluster pass
(shard.cluster_pass_sharded); rank 0 prints the totals over all ranks.

    torchrun --nproc-per-node 2 -m aletsch_b200.run --clusters a.bam b.bam c.bam
"""
import argparse
import json
import os
import sys
import time

import numpy as np

from .clusters import cluster_pass, device_batches
from . import gpu as G
from . import hostlib as H

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
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return _sharded(args, lt)
    t0 = time.time()
    recs, chrom_len = [], None
    for path in args.bams:
        r, cl = H.read_bam(path)
        if chrom_len is not None and not np.array_equal(cl, chrom_len):
            raise SystemExit("%s: reference dictionary differs from the first file's" % path)
        chrom_len = cl
        recs.append(r)
        print("%s: %d records" % (path, r["n"]), file=sys.stderr)
        if lt is None:
            pv = H.infer_library_type(r, H.default_packer_params(H.UNSTRANDED))
            lt = pv["library_type"]
            print("inferred library type %d from %s: %s" % (lt, path, pv), file=sys.stderr)
    batch = H.pack(recs, H.default_packer_params(lt), chrom_len=None if args.whole_file else chrom_len, region_length=REGION)
    t1 = time.time()
    gp = G.default_params(library_type=lt, max_group_size=args.max_group_size, min_grouping_similarity=args.min_grouping_similarity)
    ctx = G.Context(args.device)
    out = {"samples": len(recs), "bundles": batch.n_bundles, "decode_pack_s": round(t1 - t0, 3)}
    parts = device_batches(batch)
    if len(parts) > 1:
        # more than one device batch (include/aletsch_gpu.h, BATCHING RULE): cut by position; with --clusters the bundles are
        # regrouped on the device by cross-sample cluster (clusters.cluster_pass), else every part runs on its own
        out["device_batches"] = len(parts)
        if args.clusters:
            srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
            res = cluster_pass(ctx, parts, srcs, gp)
            for s in srcs:
                s.free()
            out["clusters_of_bundles"] = sum(len(c) for c in res.clusters)
            bts = res.batches
        else:
            def bridged(p):
                bt = ctx.upload(p.view(), keepalive=p)
                bt.bridge_all(gp)
                return bt
            bts = (bridged(p) for p in parts)
        tot, phases = {}, 0
        for bt in bts:
            bt.graph(gp)
            phases += int(sum(len(p["phase_cnt"]) for p in bt.phase_set()))
            for n, v in bt.counts().items():
                tot[n] = tot.get(n, 0) + v
            bt.free()
        out.update(tot)
        out["distinct_phases"] = phases
        out["device_s"] = round(time.time() - t1, 3)
        ctx.close()
        print(json.dumps(out))
        return 0
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.bridge_all(gp)
    if args.clusters and batch.n_bundles:
        off, val = bt.fetch_splices()
        a = batch.a
        # bundle groups: (chromosome, 1 Mb region of the bundle's first hit, bundle strand).  The strand is the one
        # bundle_base::compute_strand leaves (for unstranded libraries the majority of the XS tags: '+', '-' and '.' bundles are
        # grouped separately, meta/incubator.cc:526-540).  The region is the NOMINAL one: the reference files a bundle under the
        # region-table entry its generator::resolve ran for, which reaches past the 1 Mb multiple until a gap wider than
        # min_bundle_gap (rnacore/sample_profile.cc:167-252), so a bundle starting just behind a boundary inside such a run joins
        # the previous group there and the next one here; and bundle_group::remove_duplicates (meta/bundle_group.cc:58-91: '+'
        # bundles that end at or before the previous region's end1 are emptied) is not applied.  This tool is a usage example of
        # the ABI, not a reference-equivalent scheduler: the incubator stays on the host (BASELINE.json: north_star).
        from .shard import bundle_region_keys
        key = bundle_region_keys(batch)
        order = np.lexsort((np.arange(batch.n_bundles), a["bundle_sample"], key))
        cuts = np.nonzero(np.diff(key[order]))[0] + 1
        groups = [g for g in np.split(order, cuts) if len(g)]
        goff = np.zeros(len(groups) + 1, np.int32)
        np.cumsum([len(g) for g in groups], out=goff[1:])
        loff, lval = G.reorder_lists(off, val, order)
        cl_of, ncl = G.group_resolve_arrays(ctx, goff, loff, lval, gp)
        clusters = []
        for gi in range(len(groups)):
            byc = {}
            for l in range(int(goff[gi]), int(goff[gi + 1])):
                byc.setdefault(int(cl_of[l]), []).append(int(order[l]))
            clusters.extend(v for _, v in sorted(byc.items()) if len(v) >= 2)
        if clusters:
            bt.group_bridge(clusters, gp)
        out["region_groups"] = len(groups)
        out["clusters_of_bundles"] = len(clusters)
    bt.graph(gp)
    phases = bt.phase_set()
    out.update(bt.counts())
    out["distinct_phases"] = int(sum(len(p["phase_cnt"]) for p in phases))
    out["device_s"] = round(time.time() - t1, 3)
    bt.free()
    ctx.close()
    print(json.dumps(out))
    return 0


def _sharded(args, lt):
    """the run with one process per GPU: samples dealt to ranks by file index, the cluster pass over all of them"""
    import torch
    import torch.distributed as dist
    from .shard import bundle_keys, cluster_pass_sharded
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        rank, world = dist.get_rank(), dist.get_world_size()
        t0 = time.time()
        mine = [i for i in range(len(args.bams)) if i % world == rank]
        recs, chrom_len = [], None
        for i in mine:
            r, cl = H.read_bam(args.bams[i])
            if chrom_len is not None and not np.array_equal(cl, chrom_len):
                raise SystemExit("%s: reference dictionary differs from the first file's" % args.bams[i])
            chrom_len = cl
            recs.append(r)
            print("rank %d: %s: %d records" % (rank, args.bams[i], r["n"]), file=sys.stderr)
        dicts = [None] * world
        dist.all_gather_object(dicts, None if chrom_len is None else [int(x) for x in chrom_len])
        ref = dicts[0]                   # rank 0 holds file 0
        for r, d in enumerate(dicts):
            if d is not None and d != ref:      # file r is the first file of rank r
                raise SystemExit("%s: reference dictionary differs from the first file's" % args.bams[r])
        if lt is None:
            got = [None]
            if rank == 0:
                pv = H.infer_library_type(recs[0], H.default_packer_params(H.UNSTRANDED))
                got[0] = pv["library_type"]
                print("inferred library type %d from %s: %s" % (got[0], args.bams[0], pv), file=sys.stderr)
            dist.broadcast_object_list(got, src=0)
            lt = got[0]
        batch = H.pack(recs, H.default_packer_params(lt), sample_ids=mine, chrom_len=None if args.whole_file else np.array(ref, np.int32),
                       region_length=REGION)
        t1 = time.time()
        gp = G.default_params(library_type=lt, max_group_size=args.max_group_size, min_grouping_similarity=args.min_grouping_similarity)
        ctx = G.Context(local)
        parts = device_batches(batch) if batch.n_bundles else []
        out = {"bundles": batch.n_bundles, "device_batches": len(parts), "clusters_of_bundles": 0}
        if args.clusters:
            srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
            res = cluster_pass_sharded(ctx, parts, srcs, bundle_keys(batch), gp)
            for s in srcs:
                s.free()
            out["clusters_of_bundles"] = sum(len(c) for c in res.clusters)
            bts = res.batches
        else:
            def bridged(p):
                bt = ctx.upload(p.view(), keepalive=p)
                bt.bridge_all(gp)
                return bt
            bts = (bridged(p) for p in parts)
        phases = 0
        for bt in bts:
            bt.graph(gp)
            phases += int(sum(len(p["phase_cnt"]) for p in bt.phase_set()))
            for n, v in bt.counts().items():
                out[n] = out.get(n, 0) + v
            bt.free()
        out["distinct_phases"] = phases
        out["decode_pack_s"], out["device_s"] = t1 - t0, time.time() - t1
        ctx.close()
        every = [None] * world
        dist.all_gather_object(every, out)
        if rank == 0:
            tot = {"samples": len(args.bams)}
            for o in every:
                for n, v in o.items():
                    tot[n] = max(tot.get(n, 0), v) if n.endswith("_s") else tot.get(n, 0) + v
            tot["decode_pack_s"], tot["device_s"] = round(tot["decode_pack_s"], 3), round(tot["device_s"], 3)
            tot["ranks"] = world
            print(json.dumps(tot))
    finally:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
