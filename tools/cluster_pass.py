#!/usr/bin/env python
"""tools/cluster_pass.py -- the cross-sample cluster pass (aletsch_b200/clusters.py) on bench.py's workloads, on the GPU.

  python tools/cluster_pass.py --config 2                 the job cut by the batching rule (configs[2]: 4 device batches)
  python tools/cluster_pass.py --config 1 --cut 3 --check a forced 3-way cut, compared with the single-batch run

Reports per phase the host-clock time around synchronised work after a warm-up pass (source evidence, stage 5, plan, gather, and per
output batch bridge_all, group_bridge, group_support); the gather kernels' time from the per-kernel events (agpu_profile_enable),
their algorithmic bytes (per hit 34 B read + 34 B written: 4 x i32, 2 x u8, u64 qid, u32 cigar_off; per CIGAR operation 4 B read + 4
B written) and GB/s; the host route it replaces (PackedBatch.select + compact form + agpu_batch_upload_packed of the same output
batches, from pageable host memory); and, with --check, the count of bundles whose digests (bench.view_digests) and of clusters whose
support rows differ from the single-batch run.  Prints one JSON line; progress goes to stderr."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench                                                   # noqa: E402
from aletsch_b200 import clusters as CL                        # noqa: E402
from aletsch_b200 import gpu as G                              # noqa: E402
from aletsch_b200 import hostlib as H                          # noqa: E402

HIT_BYTES = 2 * 34
OP_BYTES = 2 * 4
COPY_KERNELS = ("k_gather_hits", "k_gather_cigar")


def card():
    """name, power limit and maximum SM clock of the card (read-only query)"""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "unknown"
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def copy_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, ValueError, KeyError):
        return 6543.1, "measured B200 copy peak named in BASELINE.md"


def cluster_pass(ctx, parts, srcs, gp, support, times=None):
    for s in srcs:
        s.reset()
    return CL.cluster_pass(ctx, parts, srcs, gp, support=support, times=times)


def single_batch(ctx, batch, gp, support):
    """the same job as ONE device batch: bridge_all, stage 5 over the region groups, group_bridge, group_support"""
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.bridge_all(gp)
    off, val = bt.fetch_splices()
    groups = bench.region_groups(batch)
    order = np.concatenate(groups)
    goff = np.concatenate([[0], np.cumsum([len(g) for g in groups])]).astype(np.int32)
    loff, lval = G.reorder_lists(off, val, order)
    cl_of, _ = G.group_resolve_arrays(ctx, goff, loff, lval, gp)
    multi = []
    for gi in range(len(groups)):
        byc = {}
        for l in range(int(goff[gi]), int(goff[gi + 1])):
            byc.setdefault(int(cl_of[l]), []).append(int(order[l]))
        multi.extend(v for _, v in sorted(byc.items()) if len(v) >= 2)
    if multi:
        bt.group_bridge(multi, gp)
    rows = CL._group_support(bt, multi, gp) if (support and multi) else []
    return bt, multi, rows


def same_rows(a, b):
    if sorted(a) != sorted(b):
        return False
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.shape != y.shape:
            return False
        if x.dtype == np.float64:
            if not np.allclose(x, y, rtol=1e-9, atol=0):
                return False
        elif not np.array_equal(x, y):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=1)
    ap.add_argument("--scale", type=float, default=None)
    ap.add_argument("--cut", type=int, default=0, help="cut the job into this many parts instead of by the batching rule")
    ap.add_argument("--check", action="store_true", help="compare with the single-batch run (the job must fit one device batch)")
    ap.add_argument("--no-support", action="store_true")
    args = ap.parse_args()
    support = not args.no_support
    cfg = bench.config_of(args)
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
    batch, _ = bench.build_workload(cfg, 0, max(2, ncpu))
    parts = batch.split(args.cut) if args.cut > 1 else bench.device_batches(batch)
    gp = G.default_params(library_type=cfg["library_type"], min_junction_support=cfg.get("min_junction_support", 1), **cfg["group"])
    ctx = G.Context(0)
    sctx = [G.Context(0) for _ in parts]
    srcs = [c.upload(p.view(), keepalive=p) for c, p in zip(sctx, parts)]
    out = {"config": args.config, "card": card(), "bundles": batch.n_bundles, "hits": batch.n_hits, "cigar_ops": batch.n_cigar,
           "source_batches": len(parts), "cut": "forced %d-way" % args.cut if args.cut > 1 else "batching rule"}

    # bridged pairs of the per-bundle pass alone, on the sources: the group pass adds to these
    per_bundle_bridged = 0
    for s in srcs:
        s.bridge_all(gp)
        per_bundle_bridged += int(s.bundle_counts()[:, 3].sum())

    bench.log("[cluster_pass] warm-up pass")
    cluster_pass(ctx, parts, srcs, gp, support).free()
    bench.log("[cluster_pass] timed pass")
    times = {}
    t0 = time.perf_counter()
    res = cluster_pass(ctx, parts, srcs, gp, support, times)
    total_s = time.perf_counter() - t0
    multi = [c for cl in res.clusters for c in cl]
    bridged = int(sum(int(b.bundle_counts()[:, 3].sum()) for b in res.batches))
    cnt = [b.counts() for b in res.batches]
    out_hits, out_ops = sum(c["hits"] for c in cnt), sum(c["cigar_ops"] for c in cnt)
    out.update({"output_batches": len(res.batches), "stage5_clusters": res.n_clusters, "clusters": len(multi),
                "member_bundles": int(sum(len(c) for c in multi)), "bridged_per_bundle_pass": per_bundle_bridged,
                "bridged_pairs_added_by_group_pass": bridged - per_bundle_bridged,
                "seconds": {k: (round(v, 4) if not isinstance(v, list) else [round(x, 4) for x in v]) for k, v in times.items()},
                "seconds_total": round(total_s, 4)})

    # the gather kernels alone, timed by the context's per-kernel events
    ctx.profile(True)
    ctx.profile_reset()
    for o in res.origin:
        ctx.gather(srcs, o[:, :2]).free()
    prof = {k: v for k, v in ctx.profile_read().items()}
    ctx.profile(False)
    copy_ms = sum(prof.get(k, (0.0, 0))[0] for k in COPY_KERNELS)
    nbytes = HIT_BYTES * out_hits + OP_BYTES * out_ops
    peak, peak_src = copy_peak()
    gbs = nbytes / (copy_ms / 1e3) / 1e9 if copy_ms > 0 else None
    out["gather"] = {"kernels_ms": {k: round(v[0], 4) for k, v in prof.items()}, "copy_kernels_ms": round(copy_ms, 4),
                     "algorithmic_bytes": nbytes, "copy_gbs": gbs, "copy_peak_gbs": peak, "copy_peak_source": peak_src,
                     "share_of_copy_peak": gbs / peak if gbs else None,
                     "host_seconds": round(times.get("gather", 0.0), 4)}

    # the route it replaces: host select + compact form + packed upload of the same output batches
    t_sel = t_pack = t_up = 0.0
    for o in res.origin:
        ta = time.perf_counter()
        sel = batch.select(o[:, 2])
        tb = time.perf_counter()
        arr = sel.compact()
        tc = time.perf_counter()
        b = ctx.upload(H.compact_struct(arr, sel.n_cigar), keepalive=(arr, sel))
        ctx.sync()
        td = time.perf_counter()
        b.free()
        t_sel, t_pack, t_up = t_sel + tb - ta, t_pack + tc - tb, t_up + td - tc
    out["host_select_upload_seconds"] = {"select": round(t_sel, 4), "compact": round(t_pack, 4), "upload_packed": round(t_up, 4),
                                         "total": round(t_sel + t_pack + t_up, 4)}

    if args.check:
        bench.log("[cluster_pass] single-batch run")
        got_dig = np.zeros((batch.n_bundles, 3), np.uint64)
        for b, o in zip(res.batches, res.origin):
            got_dig[o[:, 2]] = bench.view_digests(b.results(G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS), len(o))
        got_rows = [d for s in (res.support or []) for d in s]
        got_multi = [[int(o[m, 2]) for m in c] for o, cl in zip(res.origin, res.clusters) for c in cl]
        res.free()
        for s in srcs:
            s.free()
        srcs = []
        bt, want_multi, want_rows = single_batch(ctx, batch, gp, support)
        want_dig = bench.view_digests(bt.results(G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS), batch.n_bundles)
        bt.free()
        out["check"] = {"clusters_identical": got_multi == want_multi,
                        "mismatching_bundles": int((got_dig != want_dig).any(axis=1).sum()),
                        "support_clusters_compared": len(want_rows),
                        "mismatching_support_clusters": (sum(not same_rows(a, b) for a, b in zip(want_rows, got_rows))
                                                         + abs(len(want_rows) - len(got_rows)))}
    else:
        res.free()
    for s in srcs:
        s.free()
    for c in sctx + [ctx]:
        c.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
