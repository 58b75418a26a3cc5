#!/usr/bin/env python
"""bench.py -- throughput of the per-bundle read-evidence hot path (bundle::bridge, meta/bundle.cc:55-88)
on synthetic sorted-BAM records of BASELINE.json's shape.

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference ...                     the reference's own C++ (oracle/_ref) on the host cores

Workload at N = 1: configs[1] of BASELINE.json -- 10 synthetic paired_end samples x 5M pairs on one 100 Mb
chromosome, bridging on.  For N > 1 every rank gets its own chromosome of that shape (weak scaling; bundles
are independent, there is no data-path collective).  A step = one pass of the hot path over the batch:
evidence (CIGAR -> coverage / chains) -> mate pairing -> splice graphs -> paired-read clusters -> bridging DP +
vote -> update_bridges.  Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from aletsch_b200 import hostlib as H   # noqa: E402

SEED0 = 20260101             # synth-v1: seed = SEED0 + config index (SURVEY.md section 8d)

# BASELINE.json configs.  `templates` = pairs / reads per sample PER GPU; `n_chrom` chromosomes of `chrom_len` per GPU.
# configs[2] is the 8-GPU job (100 samples x 20M pairs over a 24-chromosome genome): each GPU owns 24 / 8 = 3 chromosomes, i.e.
# 20M / 8 = 2.5M pairs per sample; `scale` (default below) shrinks the depth so that generation + run stay within minutes.
CONFIGS = {
    0: dict(what="1 synthetic paired_end sample x %d pairs, 1 chromosome of %d bp per GPU, bridging on", mode="paired", samples=1,
            templates=2_000_000, n_chrom=1, chrom_len=100_000_000, scale=1.0, group=dict(max_group_size=200, min_grouping_similarity=0.10),
            group_str="-c 200 -s 0.1 (defaults)"),
    1: dict(what="10 synthetic paired_end samples x %d pairs, 1 chromosome of %d bp per GPU, bridging on", mode="paired", samples=10,
            templates=5_000_000, n_chrom=1, chrom_len=100_000_000, scale=1.0, group=dict(max_group_size=20, min_grouping_similarity=0.2),
            group_str="-c 20 -s 0.2"),
    2: dict(what="100 synthetic paired_end samples x %d pairs on this GPU's 3 of 24 chromosomes (%d bp each): the per-GPU shard of the "
                 "8-GPU job at depth scale", mode="paired", samples=100, templates=2_500_000, n_chrom=3, chrom_len=100_000_000, scale=0.1,
            group=dict(max_group_size=200, min_grouping_similarity=0.10), group_str="-c 200 -s 0.1 (defaults)"),
    3: dict(what="single-cell style: 1000 cells x %d single_end reads, 1 chromosome of %d bp per GPU, each cell expressing 10%% of the genes",
            mode="single", samples=1000, templates=200_000, n_chrom=1, chrom_len=100_000_000, scale=1.0, expressed_fraction=0.1,
            group=dict(max_group_size=2000, min_grouping_similarity=0.10), group_str="-c 2000 -s 0.1"),
    4: dict(what="20 synthetic long-read samples x %d reads (ont preset: min_junction_support 2), 1 chromosome of %d bp per GPU",
            mode="long", samples=20, templates=500_000, n_chrom=1, chrom_len=100_000_000, scale=1.0, min_junction_support=2,
            group=dict(max_group_size=200, min_grouping_similarity=0.10), group_str="-c 200 -s 0.1 (defaults)"),
}
MAX_BATCH_SPAN = 3_000_000_000     # window positions per device batch: the ABI's coverage index is 32-bit (AGPU_ERR_CAPACITY above 2^32)
MAX_BATCH_HITS = 60_000_000
E2E_CHUNK_HITS = 8_000_000
E2E_CHUNK_OPS = 32_000_000


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def config_of(args):
    c = dict(CONFIGS[args.config])
    c["scale_used"] = args.scale if args.scale is not None else c["scale"]
    c["per_sample"] = max(1000, int(c["templates"] * c["scale_used"]))
    c["mode_id"] = {"paired": H.SYNTH_PAIRED, "single": H.SYNTH_SINGLE, "long": H.SYNTH_LONG}[c["mode"]]
    c["library_type"] = H.FR_FIRST if c["mode"] == "paired" else H.UNSTRANDED
    c["seed"] = SEED0 + args.config
    return c


def workload_string(c, index):
    return "configs[%d]: " % index + c["what"] % (c["per_sample"], c["chrom_len"])


def build_workload(cfg, rank, threads):
    """records of all samples on this rank's chromosome(s), packed into one host batch of bundles"""
    t0 = time.time()
    kw = {}
    if "expressed_fraction" in cfg:
        kw["expressed_fraction"] = cfg["expressed_fraction"]
    sc = H.default_config(cfg["mode_id"], chrom_len=cfg["chrom_len"], n_chrom=cfg["n_chrom"], seed=cfg["seed"] + 1000 * rank, **kw)
    syn = H.Synth(sc)
    ns = cfg["samples"]
    recs = [None] * ns
    n_records = [0] * ns
    sem = threading.Semaphore(max(1, threads // 2))

    def guarded(k):
        with sem:
            recs[k] = syn.sample(k, cfg["per_sample"], threads=2)
            n_records[k] = recs[k]["n"]

    # a bounded number of generator threads at a time (1000 cells do not get 1000 threads)
    pending = list(range(ns))
    while pending:
        wave, pending = pending[:4 * threads], pending[4 * threads:]
        ths = [threading.Thread(target=guarded, args=(k,)) for k in wave]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    t1 = time.time()
    batch = H.pack(recs, H.default_packer_params(cfg["library_type"]))
    t2 = time.time()
    log("[bench] rank %d: %d records generated in %.1fs, packed %d bundles / %d admitted hits in %.1fs" %
        (rank, sum(n_records), t1 - t0, batch.n_bundles, batch.n_hits, t2 - t1))
    return batch, sum(n_records)


def device_batches(batch):
    """The batching rule of the ABI: one device batch holds < 2^32 coverage-window positions (the border bitmap is indexed with 32
    bits, agpu_batch_evidence returns AGPU_ERR_CAPACITY otherwise) -- cut the host batch into contiguous runs of whole bundles
    below MAX_BATCH_SPAN window positions and MAX_BATCH_HITS hits.  configs[0], [1], [4] fit one batch."""
    a = batch.a
    off = a["bundle_hit_off"]
    nb = batch.n_bundles
    if nb == 0:
        return [batch]
    first = np.minimum(off[:-1], max(batch.n_hits - 1, 0))
    last = np.maximum(off[1:] - 1, first)
    # window of a bundle: [lpos, rpos) grown to 128-base alignment; rpos may be a mate position up to 500 kb further (add_hit)
    hi = np.maximum.reduceat(np.maximum(a["rpos"], np.where((a["mpos"] > a["rpos"]) & (a["mpos"] <= a["rpos"] + 500000), a["mpos"], 0)), first) \
        if batch.n_hits else np.zeros(nb, np.int64)
    span = np.where(off[1:] > off[:-1], (hi.astype(np.int64) - a["pos"][first].astype(np.int64)) + 512, 256)
    cuts = [0]
    s = h = 0
    for k in range(nb):
        nh = int(off[k + 1] - off[k])
        if k > cuts[-1] and (s + int(span[k]) > MAX_BATCH_SPAN or h + nh > MAX_BATCH_HITS):
            cuts.append(k)
            s = h = 0
        s += int(span[k])
        h += nh
    cuts.append(nb)
    if len(cuts) == 2:
        return [batch]
    return [batch.slice(cuts[i], cuts[i + 1]) for i in range(len(cuts) - 1)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = "/tmp/agpu_clocks_%d_%d.csv" % (os.getpid(), index)

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
        return out


def algorithmic_bytes(kernel, cnt, n_cigar, n_mblocks, n_splice_pairs):
    """bytes a kernel has to read + write once per STEP (all its launches of a step together; DESIGN.md section 3),
    from the real counts of the batch"""
    Hh, S, F, C = cnt["hits"], cnt["segments"], cnt["fragments"], cnt["clusters"]
    J, V, E, NBD, M = cnt["junctions"], cnt["vertices"], cnt["edges"], cnt["borders"], cnt["cluster_members"]
    Mbig = cnt.get("big_group_members", 0)
    kernel = kernel.replace("(side)", "")
    kernel = {"k_hit_cigar_warp": "k_hit_cigar", "k_cov_add_warp": "k_cov_add"}.get(kernel, kernel)      # the warp-per-hit walks of long CIGARs move the same bytes
    if kernel == "k_hit_cigar":
        # in: pos, rpos, cigar_off (12 B/hit) + CIGAR ops; out: nspl, hash, bundle id (16 B/hit) + splice coordinates
        # + one read-modify-write of a 4-byte bitmap word per block end
        return Hh * (12 + 16) + 4 * n_cigar + 8 * n_splice_pairs + 16 * n_mblocks
    if kernel == "k_cov_add":
        # in: pos, cigar_off, bundle id (12 B/hit) + CIGAR ops; per block end a bitmap word, a rank word and a 4-byte RMW
        return Hh * 12 + 4 * n_cigar + 2 * n_mblocks * (4 + 4 + 8)
    if kernel == "k_pair_probe":
        # per hit: qid (8) + pos, mpos, isize (12) + bundle id (4) in, candidate word (4) out; one want[] counter RMW (8) per mate found
        return Hh * (8 + 12 + 4 + 4) + 2 * F * 8
    if kernel == "k_pair_decide":
        # per hit the candidate word (4); per paired hit its own and its mate's want / candidate words (16) in, mate (4) out
        return Hh * 4 + 2 * F * (16 + 4)
    if kernel == "k_hcst_insert":
        return Hh * (4 + 8 + 4 + 1 + 8) + 8 * n_splice_pairs
    if kernel == "k_frag_align":
        return F * (12 + 2 * (4 + 4 + 4) + 16 + 8 + 4)
    if kernel == "k_graph_build":
        # in: segments (12 B) and chain coordinates / counts; out: junctions (9 ints), partial exons (6 ints + 3 doubles),
        # vertices (6 ints + 3 doubles), edges (3 ints + 1 double), both adjacency tables
        return 12 * S + 4 * cnt["splice_ints"] + 12 * cnt["chains"] + 36 * J + 48 * (V - 2 * cnt.get("bundles", 0)) + 48 * V + 20 * E + 16 * E + 8 * V
    if kernel == "k_vote":
        # both passes: per cluster vp1, vp2, bundle, two chain ids, two bounds, pier (32 B) in, 8 result words (36 B) out, the pick
        # and two offsets (20 B) back in; the coordinates of the chosen chain / whole read and written once
        return C * (32 + 36 + 20) + 8 * cnt["bridge_whole_ints"] + 8 * cnt["bridge_chain_ints"]
    # the two partition kernels split the cluster members between them: the groups of more than 16 fragments (Mbig members) go
    # to the warp kernel, the rest to the thread-per-group kernel; h1 / h2, four keys, member + cluster flag out = 32 B/member
    if kernel == "k_group_partition_warp":
        return Mbig * (8 + 16 + 8)
    if kernel == "k_group_partition":
        return (M - Mbig) * (8 + 16 + 8)
    if kernel == "k_update":
        return 2 * (C * 24 + M * (4 + 8 + 8 + 2)) + M * 4 + cnt["bridged"] * 20
    return None


def step_bytes(cnt, n_cigar):
    """whole-step algorithmic bytes (stages 1-3 of SURVEY.md section 8(d) + the graph / cluster headers from the real counts).
    `survey`: the formula as the survey wrote it, with a per-base difference array (8.25 B per base of bundle span L).
    `layout`: the same with this implementation's border-compacted coverage map (3 bits per base for the border bitmap + 16 B per
    border instead of the per-base array) -- the smaller, stricter denominator."""
    Hh, S, F, C, L = cnt["hits"], cnt["segments"], cnt["fragments"], cnt["clusters"], cnt["span"]
    J, V, E, NBD, M = cnt["junctions"], cnt["vertices"], cnt["edges"], cnt["borders"], cnt["cluster_members"]
    common = 76 * Hh + 4 * n_cigar + 12 * S + 16 * J + 4 * cnt["splice_ints"] + 48 * max(V - 2 * cnt.get("bundles", 0), 0) + 56 * V + 20 * E \
        + 12 * F + 16 * F + 32 * C + 4 * M + 8 * cnt["bridge_whole_ints"] + 8 * cnt["bridge_chain_ints"]
    return {"survey": common + 8.25 * L, "layout": common + 3 * L / 8 + 16 * NBD}


def gpu_params(cfg, G):
    return G.default_params(library_type=cfg["library_type"], min_junction_support=cfg.get("min_junction_support", 1))


FIELDS = ["bundle_hit_off", "bundle_tid", "bundle_sample", "pos", "rpos", "mpos", "isize", "flag", "strand", "xs", "qid", "cigar_off", "cigar"]


def _tview(a):
    return a.view(np.int64) if a.dtype == np.uint64 else (a.view(np.int32) if a.dtype == np.uint32 else (a.view(np.int16) if a.dtype == np.uint16 else a))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from aletsch_b200 import gpu as G

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    # several ranks on one box: keep this rank's threads and pinned buffers on the NUMA node its GPU hangs off (before anything
    # is pinned); a single rank keeps every core, its cpu_baseline leg uses them
    numa_bind = {"bound": False, "why": "single rank"}
    if world > 1:
        from aletsch_b200 import affinity
        numa_bind = affinity.bind_to_device(local)
        print("[bench] rank %d: NUMA binding %s" % (rank, numa_bind), file=sys.stderr)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
    cfg = config_of(args)
    batch, n_records = build_workload(cfg, rank, max(2, ncpu // max(1, world)))
    parts = device_batches(batch)
    gp = gpu_params(cfg, G)
    stream = torch.cuda.current_stream()

    # ---- device-resident timing: inputs already in HBM, a step = (reset + bridge_all) over every device batch ---------------
    ctxs, bts, devs = [], [], []
    for part in parts:
        dev = {f: torch.from_numpy(_tview(part.a[f])).to("cuda") for f in FIELDS}
        b = H.BatchIn()
        b.n_bundles, b.n_hits, b.n_cigar = part.n_bundles, part.n_hits, part.n_cigar
        for f in FIELDS:
            setattr(b, f, dev[f].data_ptr())
        c = G.Context(local, stream=stream.cuda_stream)
        ctxs.append(c)
        bts.append(c.adopt(b, keepalive=dev))
        devs.append(dev)
    torch.cuda.synchronize()
    ctx, bt = ctxs[0], bts[0]

    n_hits = batch.n_hits
    ops = batch.a["cigar"] & 0xF
    n_mblocks = int(np.count_nonzero(ops == 0))
    n_cigar = int(batch.n_cigar)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        for x in bts:
            x.reset()
            x.bridge_all(gp)

    def sum_counts():
        tot = {}
        for x in bts:
            for k, v in x.counts().items():
                tot[k] = tot.get(k, 0) + v
        return tot

    for _ in range(args.warmup):
        one_step()
    for c in ctxs:
        c.sync()
    launches0 = sum(c.launches for c in ctxs)
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        one_step()
    e1.record(stream)
    barrier()
    ms_dev = e0.elapsed_time(e1)
    launches = sum(c.launches for c in ctxs) - launches0
    # the same K steps again with CUDA events around every kernel launch (per-kernel durations for the roofline; the
    # event records cost ~2% so they stay out of the region `value` is taken from)
    for c in ctxs:
        c.profile(True)
        c.profile_reset()
    ep0, ep1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ep0.record(stream)
    for _ in range(args.steps):
        one_step()
    ep1.record(stream)
    barrier()
    ms_prof = ep0.elapsed_time(ep1)
    clk = clocks.stop()
    prof = {}
    for c in ctxs:
        for name, (ms, cnt) in c.profile_read().items():
            m = prof.setdefault(name, [0.0, 0])
            m[0] += ms
            m[1] += cnt
        c.profile(False)
    counts = sum_counts()
    per_bundle = np.concatenate([x.bundle_counts() for x in bts]) if bts else np.zeros((0, 4), np.int64)   # [NB, 4]: segments, fragments, clusters, bridged
    # digests of the result arrays of every bundle (for the full-size cross-check against the reference run, cpu_baseline)
    digests = None
    if not args.no_cpu_baseline and rank == 0:
        digests = np.concatenate([view_digests(x.results(G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS), x_part.n_bundles)
                                  for x, x_part in zip(bts, parts)]) if bts else np.zeros((0, 3), np.uint64)
    # the event-profiled repeat above ran the same reset + bridge_all on the same inputs: the device holds the last timed step's results
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bts, parts, per_bundle, counts)
    stage5 = stage5_gpu(ctx, bts, batch, parts, cfg, args) if not args.no_stage5 else None
    single = len(parts) == 1
    group_leg = group_bridge_gpu(ctx, bt, gp, stage5_gpu.clusters, args) if (stage5 is not None and single and cfg["mode"] == "paired") else None
    support_leg = support_gpu(ctx, bt, gp, stage5_gpu.clusters, args) if (stage5 is not None and single) else None
    phase_leg = phase_set_gpu(bts, gp, args) if stage5 is not None else None
    for x in bts:
        x.free()
    for c in ctxs:
        c.close()
    del devs, bts, ctxs

    # ---- end to end: pinned host buffers -> upload -> bridge_all -> EVERY result structure back in host memory ----------------
    # the public call: aletsch_b200.pipeline.Pipeline.run over the batch cut into contiguous sub-batches, a few host threads
    # with one CUDA stream each, so the H2D copy of one sub-batch overlaps the kernels (and the D2H copies) of another
    from aletsch_b200.pipeline import Pipeline
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    # sub-batches of at most ~E2E_CHUNK_HITS hits: each of the pool's contexts keeps an arena as large as the hungriest sub-batch
    # it has seen, so the sub-batch size bounds the device memory of the pipeline (2 x streams contexts)
    chunks = []
    for part in parts:
        per_part = max(1, -(-args.chunks // len(parts)), -(-part.n_hits // E2E_CHUNK_HITS), -(-part.n_cigar // E2E_CHUNK_OPS))
        chunks.extend(part.split(per_part))
    views = []
    h2d_bytes = 0
    for ch in chunks:
        pin = {}
        ch.a["bundle_strand"] = np.ascontiguousarray(ch.a["strand"][np.minimum(ch.a["bundle_hit_off"][:-1], max(ch.n_hits - 1, 0))])
        if args.upload == "compact":
            # the compact link format (agpu_batch_packed): 16-bit position deltas / mate offsets / insert sizes / CIGAR units
            # with escape lists, decoded on the device into the arrays of the plain upload (include/aletsch_gpu.h)
            arrays = ch.compact()
            for f, a in arrays.items():
                v = a.view(np.int64) if a.dtype == np.uint64 else (a.view(np.int16) if a.dtype == np.uint16 else a)
                pin[f] = torch.from_numpy(np.ascontiguousarray(v)).pin_memory()
                h2d_bytes += pin[f].numel() * pin[f].element_size()
            views.append((H.compact_struct(pin, ch.n_cigar, ptr=lambda t: t.data_ptr()), pin))
            continue
        # lean upload: flag[] is never read on the device, rpos[] is re-derived from the CIGAR there, and the strand that all
        # hits of a bundle share goes up once per bundle (agpu_batch_in: rpos / flag / strand may be NULL)
        lean = [f for f in FIELDS if f not in ("rpos", "flag", "strand")] + ["bundle_strand"]
        for f in lean:
            pin[f] = torch.from_numpy(_tview(ch.a[f])).pin_memory()
            h2d_bytes += pin[f].numel() * pin[f].element_size()
        b = H.BatchIn()
        b.n_bundles, b.n_hits, b.n_cigar = ch.n_bundles, ch.n_hits, ch.n_cigar
        for f in lean:
            setattr(b, f, pin[f].data_ptr())
        views.append((b, pin))
    what = {"full": G.RESULT_ALL, "bundle": G.RESULT_EVIDENCE | G.RESULT_FRAGMENTS, "counts": 0}[args.results]
    pipe = Pipeline(local, n_streams=args.streams, prefetch=not args.no_prefetch)
    for _ in range(min(args.warmup, 2)):
        pipe.run(views, gp, results=what)
    pipe.sync()
    barrier()
    launches_e2e0 = pipe.launches
    syncs_e2e0 = pipe.syncs
    if os.environ.get("AGPU_PIPE_PROFILE"):        # diagnosis: per-kernel CUDA-event times inside the pipelined run
        for c in pipe.ctxs:
            c.profile(True)
            c.profile_reset()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    # all K steps' sub-batches go through the stream pool back to back (every step uploads its inputs again and brings its
    # results back; there is no barrier between steps, the K steps are bracketed as a whole)
    res = pipe.run(views * args.steps, gp, results=what)
    pipe.sync()
    e3.record(stream)
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    d2h_bytes = sum(r["d2h_bytes"] for r in res) / args.steps + 18 * 8 * len(views)     # result views + the counter struct of every sub-batch
    launches_e2e = pipe.launches - launches_e2e0
    syncs_e2e = pipe.syncs - syncs_e2e0
    assert sum(r["hits"] for r in res) == n_hits * args.steps and sum(r["bridged"] for r in res) == counts["bridged"] * args.steps, "pipelined result differs"
    # one more pass, untimed: how long the reference-side adapter input (graph view) of every sub-batch takes to rebuild is the
    # host's business (integration/adapter.cc); here only the device -> host part is timed.  Per-view split of the traffic:
    if os.environ.get("AGPU_PIPE_PROFILE"):
        acc = {}
        for c in pipe.ctxs:
            for name, (ms, cnt) in c.profile_read().items():
                m = acc.setdefault(name, [0.0, 0])
                m[0] += ms
                m[1] += cnt
        for name, (ms, cnt) in sorted(acc.items(), key=lambda kv: -kv[1][0])[:25]:
            log("[pipe-profile] %-28s %10.3f ms total  %6d launches  %9.3f ms/launch" % (name, ms, cnt, ms / max(cnt, 1)))
    if pipe.trace is not None:
        t00 = min(x[3] for x in pipe.trace[-4 * len(views) * args.steps:])
        for i, what, tid, a, b in pipe.trace[-4 * len(views) * args.steps:]:
            log("[trace] sub-batch %2d %-8s thread %x  %8.2f -> %8.2f ms (%7.2f)" % (i, what, tid & 0xffff, 1e3 * (a - t00), 1e3 * (b - t00), 1e3 * (b - a)))
    pipe.close()

    # ---- the path's one exchange step (world > 1): samples ingested on different ranks share their per-bundle splice signatures
    # with ONE all-gather over NCCL, after which every rank runs the identical bundle_group::resolve (aletsch_b200/shard.py).
    # Here every rank contributes the signatures of its own chromosome(s); timed on the device, max over ranks.
    collective = None
    if world > 1:
        from aletsch_b200 import shard
        cctx = G.Context(local, stream=stream.cuda_stream)
        sig_off, sig_val = [np.zeros(1, np.int64)], []
        base = 0
        for part in parts:
            dev = {f: torch.from_numpy(_tview(part.a[f])).to("cuda") for f in FIELDS}
            b = H.BatchIn()
            b.n_bundles, b.n_hits, b.n_cigar = part.n_bundles, part.n_hits, part.n_cigar
            for f in FIELDS:
                setattr(b, f, dev[f].data_ptr())
            x = cctx.adopt(b, keepalive=dev)
            x.evidence(gp)
            o, v = x.fetch_splices()
            x.free()
            sig_off.append(o[1:] + base)
            sig_val.append(v)
            base += int(o[-1]) if len(o) else 0
            del dev
        sig_off = np.concatenate(sig_off)
        sig_val = np.concatenate(sig_val) if sig_val else np.zeros(0, np.int32)
        keys = (np.int64(rank) << 40) | np.arange(batch.n_bundles, dtype=np.int64)
        regs = shard.bundle_region_keys(batch) | (np.int64(rank) << 56)
        for it in range(3):
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            t_host0 = time.perf_counter()
            got = shard.gather_packed(sig_off, sig_val, keys, regs)
            c1.record(stream)
            barrier()
            t_host = time.perf_counter() - t_host0
            ms_coll = c0.elapsed_time(c1)
        tc = torch.tensor([ms_coll, t_host * 1e3], dtype=torch.float64, device="cuda")
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        collective = {"name": "all_gather (NCCL, torch.distributed) of the per-bundle splice signatures: header + padded payload",
                      "bundles_gathered": int(len(got[0]) - 1), "signature_values": int(len(got[1])), "bytes_received_per_rank": int(got[5]),
                      "device_ms": float(tc[0]), "host_wall_ms": float(tc[1]), "timing": "CUDA events around the two collectives, max over ranks"}
        cctx.close()
        torch.cuda.empty_cache()

    # max over ranks, totals over ranks
    t = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_hits), float(counts["bridged"]), float(h2d_bytes), float(d2h_bytes)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    hits_all, bridged_all = float(tot[0]), float(tot[1])

    if rank == 0:
        steps = args.steps
        value = hits_all * steps / (ms_dev / 1e3)
        e2e_value = hits_all * steps / (ms_e2e / 1e3)
        # dominant kernel by accumulated device time
        total_k = sum(v[0] for v in prof.values())
        top = sorted(prof.items(), key=lambda kv: -kv[1][0])
        for name, (ms, cnt) in top[:48]:
            log("[bench] kernel %-26s %9.3f ms/step  (%d launches/step, %.1f%% of kernel time)" %
                (name, ms / steps, cnt // steps, 100 * ms / max(total_k, 1e-9)))
        # SURVEY section 8(d): bridged pairs / time of stage 4 + update = the bridging kernels' accumulated time (rank 0's batch)
        stage4 = ("k_bridge_vertices", "k_piers", "k_cluster_pier", "k_group_cand", "k_bridge_job_counts", "k_bridge_job_fill",
                  "k_bridge_dp_warp", "k_pier_bridges", "k_vote", "k_vote_type1", "k_vote_type2", "k_update", "k_fcst_insert", "k_merge_entries", "k_scatter_handle")
        stage4_ms = sum(ms for name, (ms, cnt) in prof.items() if name.replace("(side)", "") in stage4) / steps
        dom = None
        n_splice_pairs = int(np.count_nonzero(ops == 3))
        counts["bundles"] = batch.n_bundles
        # the dominant kernel: side-stream launches of the same kernel count with it
        merged = {}
        for name, (ms, cnt) in prof.items():
            m = merged.setdefault(name.replace("(side)", ""), [0.0, 0])
            m[0] += ms
            m[1] += cnt
        for name, (ms, cnt) in sorted(merged.items(), key=lambda kv: -kv[1][0]):
            ab = algorithmic_bytes(name, counts, n_cigar, n_mblocks, n_splice_pairs)
            if ab is not None:
                dom = (name, ms, cnt, ab)
                break
        # DRAM traffic of the dominant kernel from the committed ncu --set full capture of this build (profiles/), if any
        traffic, tf = {}, []
        try:
            import glob
            tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
            if tf:
                traffic = json.load(open(tf[-1]))
        except (OSError, ValueError):
            traffic = {}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        roof = None
        if dom:
            name, ms, cnt, ab = dom          # ab: bytes per step over all launches of the kernel in a step
            per_launch_ms = ms / cnt
            launches_per_step = cnt / steps
            achieved = ab / launches_per_step / (per_launch_ms / 1e3) / 1e9
            tk = traffic.get("kernels", {}).get(name)
            traffic_per_launch = (tk["dram_read_bytes"] + tk["dram_write_bytes"]) / tk["launches"] if tk else None
            sb = step_bytes(counts, n_cigar)
            step_s = ms_dev / steps / 1e3
            roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                    "algorithmic_bytes_per_launch": ab / launches_per_step, "ms_per_launch": per_launch_ms,
                    "launches_per_step": launches_per_step,
                    "share_of_kernel_time": ms / max(total_k, 1e-9), "ms_per_step_profiled": ms_prof / steps, "traffic": traffic_per_launch,
                    "traffic_source": os.path.basename(tf[-1]) if (tk and tf) else None,
                    # the whole step against the same peak: sum of the algorithmic bytes of all stages / ms_per_step
                    "step": {"algorithmic_bytes_survey": sb["survey"], "algorithmic_bytes_layout": sb["layout"],
                             "achieved_survey": sb["survey"] / step_s / 1e9, "achieved_layout": sb["layout"] / step_s / 1e9,
                             "frac_survey": sb["survey"] / step_s / 1e9 / peak, "frac_layout": sb["layout"] / step_s / 1e9 / peak,
                             "note": "survey = SURVEY 8(d) formula with a per-base difference array (8.25 B/base); layout = the same with the "
                                     "border-compacted coverage map this implementation stores (3 bits/base + 16 B/border)"}}
        config = reference_config(cfg, args, batch, n_records, len(parts))
        out = {"metric": "hits_per_sec", "value": value, "unit": "hits/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
               "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
               "data": "synthetic", "impl": "ours", "config": config,
               "bridged_pairs_per_sec": bridged_all * steps / (ms_dev / 1e3), "bridged_pairs_per_step": bridged_all,
               "bridged_pairs_per_sec_stage4": bridged_all / max(stage4_ms / 1e3, 1e-12), "stage4_ms_per_step": stage4_ms,
               "counts": counts, "gpu_launches": int(launches),
               "e2e": {"value": e2e_value, "unit": "hits/s", "h2d_bytes_per_step": float(tot[2]), "d2h_bytes_per_step": float(tot[3]),
                       "ms_per_step": ms_e2e / steps, "upload": args.upload, "results": args.results,
                       "results_note": {"full": "agpu_batch_results(ALL): mmap segments, hcst + hit handles, frgs, fcst + fragment handles, splice graphs, "
                                                "pereads clusters, bridge paths of every bundle in pinned host memory",
                                        "bundle": "evidence + fragments views only (what bundle::bridge leaves in bundle_base)",
                                        "counts": "counters only"}[args.results],
                       "prefetch": not args.no_prefetch, "stream_drains_per_step": syncs_e2e / steps, "sub_batches": len(views), "streams": args.streams,
                       "gpu_launches_per_step": int(launches_e2e // steps)},
               "roofline": roof, "clocks": clk, "numa_bind": numa_bind}
        if collective is not None:
            out["collective"] = collective
        if stage5 is not None:
            out["stage5"] = stage5
        if group_leg is not None:
            out["group_bridge"] = group_leg
        if support_leg is not None:
            out["support"] = support_leg
        if phase_leg is not None:
            out["phase_set"] = phase_leg
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(batch, cfg, min(10, ncpu), args.cpu_seconds, gpu_bridged=per_bundle[:, 3], gpu_digests=digests)
            if stage5 is not None:
                out["stage5"]["cpu_baseline"] = stage5_cpu(batch, cfg, min(10, ncpu), max(2.0, args.cpu_seconds / 4))
            if group_leg is not None:
                out["group_bridge"]["cpu_baseline"] = group_bridge_cpu(batch, cfg, stage5_gpu.clusters, min(10, ncpu), max(2.0, args.cpu_seconds / 4))
            if support_leg is not None:
                out["support"]["cpu_baseline"] = support_cpu(batch, cfg, stage5_gpu.clusters, min(10, ncpu), max(2.0, args.cpu_seconds / 4))
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def reference_config(cfg, args, batch=None, n_records=None, n_parts=None):
    """the `config` both arms print, key for key and value for value (the driver compares them): workload string, generator and
    seed, and what the generator + packer made of it on rank 0"""
    c = {"workload": workload_string(cfg, args.config), "generator": "synth-v1 seed %d" % cfg["seed"], "scale": cfg["scale_used"],
         "samples": cfg["samples"], "templates_per_sample_per_gpu": cfg["per_sample"], "chromosomes_per_gpu": cfg["n_chrom"]}
    if batch is not None:
        plain = sum(batch.a[f].nbytes for f in FIELDS)
        c.update({"records_per_gpu": int(n_records), "admitted_hits_per_gpu": int(batch.n_hits), "bundles_per_gpu": int(batch.n_bundles),
                  "device_batches": int(n_parts if n_parts is not None else len(device_batches(batch))),
                  "l2": "no flush: a step reads %.2f GB of plain input arrays and several GB of derived state, far more than the 126 MB L2" % (plain / 1e9)})
    return c


REGION = 1_000_000      # region_partition_length (util/parameters.cc:42)


def region_groups(batch):
    """bundle groups as the reference forms them: all samples' bundles of one (chromosome, 1 Mb region, strand)
    (meta/incubator.cc:312-314, :461-471), members in (sample, bundle) order"""
    a = batch.a
    off = a["bundle_hit_off"]
    first = np.minimum(off[:-1], max(batch.n_hits - 1, 0))
    strand = a["strand"][first].astype(np.int64)
    if batch.n_hits and np.any(strand == ord(".")):
        # unstranded libraries: the bundle's strand is the majority of its hits' XS tags (bundle_base::compute_strand,
        # rnacore/bundle_base.cc:206-224); the reference groups '+', '-' and '.' bundles separately
        cp = np.concatenate([[0], np.cumsum(a["xs"] == ord("+"))])
        cm = np.concatenate([[0], np.cumsum(a["xs"] == ord("-"))])
        npl, nmi = cp[off[1:]] - cp[off[:-1]], cm[off[1:]] - cm[off[:-1]]
        maj = np.where(npl > nmi, ord("+"), np.where(npl < nmi, ord("-"), ord(".")))
        strand = np.where(strand == ord("."), maj, strand)
    key = (a["bundle_tid"].astype(np.int64) << 40) | ((a["pos"][first].astype(np.int64) // REGION) << 8) | strand
    order = np.lexsort((np.arange(batch.n_bundles), a["bundle_sample"], key))
    cuts = np.nonzero(np.diff(key[order]))[0] + 1
    return [g for g in np.split(order, cuts) if len(g)]


def stage5_gpu(ctx, bts, batch, parts, cfg, args):
    """bundle_group::resolve over every region group of the batch: splice signatures compacted on the device, all groups'
    pair counts in one launch (agpu_group_resolve_batch), size-capped union-find on the host; -c / -s of the config"""
    stage5_gpu.clusters = []
    import torch
    from aletsch_b200 import gpu as G
    gp5 = G.default_params(library_type=cfg["library_type"], **cfg["group"])
    groups = region_groups(batch)
    order = np.concatenate(groups) if groups else np.zeros(0, np.int64)
    group_off = np.zeros(len(groups) + 1, np.int32)
    np.cumsum([len(g) for g in groups], out=group_off[1:])
    clusters = 0
    t_all = []
    cl_of = np.zeros(0, np.int32)
    for it in range(1 + max(1, min(args.steps, 3))):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        # the bundles' splice lists from every device batch, in bundle order
        offs, vals, base = [np.zeros(1, np.int64)], [], 0
        for x in bts:
            o, v = x.fetch_splices()
            offs.append(o[1:] + base)
            vals.append(v)
            base += int(o[-1]) if len(o) else 0
        off = np.concatenate(offs)
        val = np.concatenate(vals) if vals else np.zeros(0, np.int32)
        loff, lval = G.reorder_lists(off, val, order)
        cl_of, ncl = G.group_resolve_arrays(ctx, group_off, loff, lval, gp5)
        torch.cuda.synchronize()
        if it > 0:
            t_all.append(time.perf_counter() - t0)
        clusters = int(ncl.sum())
    # the clusters with at least two bundles (input of assembler::bridge), members in gset order
    multi = []
    for gi, g in enumerate(groups):
        a, b = int(group_off[gi]), int(group_off[gi + 1])
        byc = {}
        for l in range(a, b):
            byc.setdefault(int(cl_of[l]), []).append(int(order[l]))
        multi.extend(v for _, v in sorted(byc.items()) if len(v) >= 2)
    stage5_gpu.clusters = multi
    dt = float(np.mean(t_all))
    pairs = int(sum(len(g) * (len(g) - 1) // 2 for g in groups))
    return {"bundle_groups": len(groups), "bundles": int(batch.n_bundles), "largest_group": int(max((len(g) for g in groups), default=0)),
            "pairs": pairs, "clusters": int(clusters), "ms": dt * 1e3,
            "bundles_per_sec": batch.n_bundles / dt, "pairs_per_sec": pairs / dt, "params": cfg["group_str"],
            "timing": "host wall clock around splice fetch + agpu_group_resolve_batch (device pair counts + host union-find), synchronised"}


def group_bridge_gpu(ctx, bt, gp, clusters, args):
    """assembler::bridge (meta/assembler.cc:977-1018) over the clusters stage 5 found: combined bundles, their splice graphs,
    every member re-clustered / re-bridged / updated against them.  Timed after a fresh per-bundle pass, host wall clock
    (the call ends with a stream synchronisation)."""
    import torch
    if not clusters:
        return None
    t_all = []
    extra = 0
    for it in range(1 + max(1, min(args.steps, 3))):
        bt.reset()
        bt.bridge_all(gp)
        before = int(bt.bundle_counts()[:, 3].sum())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bt.group_bridge(clusters, gp)
        torch.cuda.synchronize()
        if it > 0:
            t_all.append(time.perf_counter() - t0)
        extra = int(bt.bundle_counts()[:, 3].sum()) - before
    dt = float(np.mean(t_all))
    members = int(sum(len(c) for c in clusters))
    return {"clusters": len(clusters), "member_bundles": members, "ms": dt * 1e3, "member_bundles_per_sec": members / dt,
            "bridged_pairs_added": extra}


def support_gpu(ctx, bt, gp, clusters, args):
    """the cross-sample support features of assembler::assemble(vector<bundle*>) (meta/assembler.cc:177-373) over the clusters stage
    5 found, after the per-bundle and the group bridging: members' graphs rebuilt + revised, combined graphs rebuilt, the four
    support passes (agpu_batch_group_support); host wall clock, the call ends with a stream synchronisation"""
    import torch
    if not clusters:
        return None
    t_all = []
    for it in range(1 + max(1, min(args.steps, 3))):
        bt.reset()
        bt.bridge_all(gp)
        bt.group_bridge(clusters, gp)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bt.group_support(clusters, gp, fetch=False)
        torch.cuda.synchronize()
        if it > 0:
            t_all.append(time.perf_counter() - t0)
    rows = bt.group_support(clusters[:64], gp)
    edges = int(sum(len(d["x_sup_abd"]) for d in rows))
    multi = int(sum(int((d["x_sup_edge"].reshape(-1, 3)[:, 2] > 1).sum()) for d in rows))
    dt = float(np.mean(t_all))
    members = int(sum(len(c) for c in clusters))
    pairs = int(sum(len(c) * len(c) for c in clusters))
    return {"clusters": len(clusters), "member_bundles": members, "member_pairs": pairs, "ms": dt * 1e3, "member_bundles_per_sec": members / dt,
            "member_pairs_per_sec": pairs / dt, "first_64_clusters": {"combined_edges": edges, "edges_with_several_samples": multi}}


def support_cpu(batch, cfg, clusters, threads, budget_s):
    """the reference's own support functions driven in its order (oracle/ref_driver.cc: ref_group_support, scallop left out) on a
    bounded sample of the same clusters; per-bundle and group bridging done untimed first.  The timed call also rebuilds the
    members' and the combined graphs, like the device call, and fills the checker's result bag."""
    import orclib
    import parity
    kind = _checker_kind()
    op = _orc_params(cfg)
    sizes = np.diff(batch.a["bundle_hit_off"])
    total = int(sum(int(sizes[k]) for c in clusters for k in c))
    target_hits = int(60_000 * threads * budget_s)
    step = max(1, int(np.ceil(total / max(target_hits, 1))))
    sample = clusters[::step]
    lock = threading.Lock()
    nxt = [0]
    spent = [0.0]

    def worker():
        chk = orclib.Checker("ref" if kind == "reference" else "orc")
        L = chk.lib
        fs = getattr(L, chk.prefix + "_group_support")
        fs.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p]
        ss = getattr(L, chk.prefix + "_bundle_set_sample")
        ss.argtypes = [C.c_void_p, C.c_int]
        L.orc_bag_new.restype = C.c_void_p
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(sample):
                return
            hs = []
            for k in sample[i]:
                h = chk.new_bundle(batch.bundle(int(k)), op)
                chk.run_quiet(h, "fragments")
                chk.run_quiet(h, "bridge")
                ss(h, int(batch.a["bundle_sample"][int(k)]))
                hs.append(h)
            chk.group_bridge(hs)
            bag = L.orc_bag_new()
            arr = (C.c_void_p * len(hs))(*hs)
            t0 = time.perf_counter()
            fs(arr, len(hs), bag)
            dt = time.perf_counter() - t0
            L.orc_bag_free(bag)
            for h in hs:
                chk.free_bundle(h)
            with lock:
                spent[0] += dt
    os.environ["ORC_SUPPORT_GROUP_ONLY"] = "1"
    try:
        ths = [threading.Thread(target=worker) for _ in range(threads)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    finally:
        os.environ.pop("ORC_SUPPORT_GROUP_ONLY", None)
    members = int(sum(len(c) for c in sample))
    pairs = int(sum(len(c) * len(c) for c in sample))
    wall = spent[0] / threads
    return {"kind": kind, "cores": threads, "sample": "every %d-th cluster: %d clusters, %d member bundles" % (step, len(sample), members),
            "member_bundles_per_sec": members / max(wall, 1e-9), "member_pairs_per_sec": pairs / max(wall, 1e-9)}


def phase_set_gpu(bts, gp, args):
    """bundle_base::build_phase_set (rnacore/bundle_base.cc:338-418) for every bundle: graphs rebuilt from the bridged evidence,
    then the phasing paths; device part only (agpu_batch_phase_set ends with a stream synchronisation)"""
    import torch
    t_all, t_rv = [], []
    n_ph = n_el = n_add = n_mark = 0
    for it in range(1 + max(1, min(args.steps, 3))):
        dt = drv = 0.0
        n_ph = n_el = n_add = n_mark = 0
        for bt in bts:
            bt.reset()
            bt.bridge_all(gp)
            bt.graph(gp)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            bt._run("phase_set")
            torch.cuda.synchronize()
            dt += time.perf_counter() - t0
            # the boundary revision of the same transform(bd, gr, true) call (identify_boundaries + remove_false_boundaries)
            t0 = time.perf_counter()
            bt.revise(gp, fetch=False)
            torch.cuda.synchronize()
            drv += time.perf_counter() - t0
            if it == 0:
                continue
        if it > 0:
            t_all.append(dt)
            t_rv.append(drv)
    for bt in bts:
        ph = bt.phase_set()
        n_ph += int(sum(len(p["phase_cnt"]) for p in ph))
        n_el += int(sum(int(p["phase_cnt"].sum()) for p in ph))
        rv = bt.revise(gp)
        n_add += int(sum(len(r["rev_edge_d"]) for r in rv))
        n_mark += int(sum(int((r["rev_vert"] > 0).sum()) for r in rv))
    dt = float(np.mean(t_all))
    return {"ms": dt * 1e3, "distinct_phases": n_ph, "phase_elements": n_el, "phase_elements_per_sec": n_el / max(dt, 1e-12),
            "revise_ms": float(np.mean(t_rv)) * 1e3, "revise_edges_added": n_add, "revise_vertices_marked": n_mark}


def _checker_kind():
    import orclib
    try:
        orclib.Checker("ref")
        return "reference"
    except (OSError, FileNotFoundError):
        return "port"


def _orc_params(cfg, **kw):
    import orclib
    return orclib.default_params(library_type=cfg["library_type"], min_junction_support=cfg.get("min_junction_support", 1), **kw)


def group_bridge_cpu(batch, cfg, clusters, threads, budget_s):
    """the reference's assembler::bridge on a bounded sample of the same clusters (per-bundle bridging done untimed first)"""
    import orclib
    kind = _checker_kind()
    op = _orc_params(cfg)
    sizes = np.diff(batch.a["bundle_hit_off"])
    total = int(sum(int(sizes[k]) for c in clusters for k in c))
    target_hits = int(60_000 * threads * budget_s)
    step = max(1, int(np.ceil(total / max(target_hits, 1))))
    sample = clusters[::step]
    lock = threading.Lock()
    nxt = [0]
    spent = [0.0]
    added = [0]

    def worker():
        chk = orclib.Checker("ref" if kind == "reference" else "orc")
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(sample):
                return
            hs = [chk.new_bundle(batch.bundle(int(k)), op) for k in sample[i]]
            for h in hs:
                chk.run_quiet(h, "fragments")
                chk.run_quiet(h, "bridge")
            t0 = time.perf_counter()
            tot, _ = chk.group_bridge(hs)
            dt = time.perf_counter() - t0
            for h in hs:
                chk.free_bundle(h)
            with lock:
                spent[0] += dt
                added[0] += max(int(tot), 0)
    ths = [threading.Thread(target=worker) for _ in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    members = int(sum(len(c) for c in sample))
    wall = spent[0] / threads
    return {"kind": kind, "cores": threads, "sample": "every %d-th cluster: %d clusters, %d member bundles" % (step, len(sample), members),
            "member_bundles_per_sec": members / max(wall, 1e-9), "bridged_pairs_added": added[0],
            "note": "includes copying the checker's result arrays out (chk.group_bridge dumps the combined bundle and every member)"}


def stage5_cpu(batch, cfg, threads, budget_s):
    """the reference's bundle_group::resolve on a bounded sample of the same region groups (bundle objects built untimed)"""
    import orclib
    kind = _checker_kind()
    op = _orc_params(cfg, **cfg["group"])
    groups = region_groups(batch)
    sizes = np.diff(batch.a["bundle_hit_off"])
    target_hits = int(60_000 * threads * budget_s)          # building the bundle objects dominates; bound that
    step = max(1, int(np.ceil(sizes.sum() / max(target_hits, 1))))
    sample = groups[::step]
    lock = threading.Lock()
    nxt = [0]
    spent = [0.0]

    def worker():
        chk = orclib.Checker("ref" if kind == "reference" else "orc")
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(sample):
                return
            hs = [chk.new_bundle(batch.bundle(int(k)), op) for k in sample[i]]
            t0 = time.perf_counter()
            chk.group_resolve(hs, op)
            dt = time.perf_counter() - t0
            for h in hs:
                chk.free_bundle(h)
            with lock:
                spent[0] += dt
    # bundle_group::resolve prints per-group statistics lines (meta/bundle_group.cc:360-393): keep them off our stdout
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        ths = [threading.Thread(target=worker) for _ in range(threads)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)
    nbun = int(sum(len(g) for g in sample))
    pairs = int(sum(len(g) * (len(g) - 1) // 2 for g in sample))
    wall = spent[0] / threads            # thread-seconds inside bundle_group::resolve spread over the pool
    return {"kind": kind, "cores": threads, "sample": "every %d-th region group: %d groups, %d bundles" % (step, len(sample), nbun),
            "bundles_per_sec": nbun / max(wall, 1e-9), "pairs_per_sec": pairs / max(wall, 1e-9)}


class RefTimer:
    """oracle/_ref's timing entry (ref_driver.cc: ref_timing_*): a bounded sample of the batch's bundles; the BAM records and the
    `hit` objects are built once, BEFORE any clock; every pass then runs add_hit_intervals + build_fragments + the reference's own
    bundle::bridge() per bundle on a pool of `threads` workers (one bundle per task, like aletsch -t N) with no checker dumps."""

    def __init__(self, batch, cfg, threads, budget_s, rate=150_000, calibrate=True):
        self._build(batch, cfg, threads, budget_s, rate)
        if calibrate and self.step > 1:
            # the hits/s per core depend on the depth of the bundles: one untimed pass, then resize the sample once so that a
            # pass lasts about `budget_s`
            sec, _ = self.run()
            if sec < 0.7 * budget_s or sec > 1.5 * budget_s:
                measured = self.hits / max(sec, 1e-6) / threads
                self.close()
                self._build(batch, cfg, threads, budget_s, measured)

    def _build(self, batch, cfg, threads, budget_s, rate):
        import orclib
        self.lib = L = C.CDLL(orclib.REF_SO)
        L.ref_timing_new.restype = C.c_void_p
        L.ref_timing_new.argtypes = [C.c_int, C.c_void_p, C.POINTER(orclib.Params)]
        L.ref_timing_free.argtypes = [C.c_void_p]
        L.ref_timing_hits.restype = C.c_int64
        L.ref_timing_hits.argtypes = [C.c_void_p]
        L.ref_timing_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_void_p]
        self.threads = threads
        sizes = np.diff(batch.a["bundle_hit_off"])
        # bounded sample: every k-th bundle until the estimated work of ONE pass fits the budget (~`rate` hits/s per core)
        target_hits = int(rate * threads * budget_s)
        self.step = max(1, int(np.ceil(sizes.sum() / max(target_hits, 1))))
        self.sample = list(range(0, batch.n_bundles, self.step))
        n = len(self.sample)
        arr = (orclib.BundleIn * max(n, 1))()
        self.keep = []
        for j, k in enumerate(self.sample):
            bd = batch.bundle(k)
            arr[j].n_hits = len(bd["pos"])
            arr[j].tid = bd["tid"]
            for f in ("pos", "mpos", "isize", "flag", "strand", "xs", "qid", "cigar_off", "cigar"):
                a = np.ascontiguousarray(bd[f])
                self.keep.append(a)
                setattr(arr[j], f, a.ctypes.data)
        op = _orc_params(cfg)
        self.h = L.ref_timing_new(n, C.cast(arr, C.c_void_p), C.byref(op))
        self.keep = None          # the handle owns its records and hits now
        self.hits = int(L.ref_timing_hits(self.h))
        self.per = np.zeros(max(n, 1), np.int32)

    def run(self):
        sec, br = C.c_double(0), C.c_int64(0)
        self.lib.ref_timing_run(self.h, self.threads, C.byref(sec), C.byref(br), self.per.ctypes.data)
        return sec.value, int(br.value)

    def digests(self):
        """[n_sample, 3] uint64: ref_timing_digest (untimed) -- mmap segments, frgs, splices of every sampled bundle after bundle::bridge()"""
        self.lib.ref_timing_digest.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        d = np.zeros((max(len(self.sample), 1), 3), np.uint64)
        self.lib.ref_timing_digest(self.h, self.threads, d.ctypes.data)
        return d[:len(self.sample)]

    def describe(self, sec):
        return "every %d-th bundle of the same batch: %d bundles, %d hits, %.2f s per pass" % (self.step, len(self.sample), self.hits, sec)

    def close(self):
        if self.h:
            self.lib.ref_timing_free(self.h)
            self.h = None


def _mix_rows(a, b, c, j):
    """row_digest of oracle/ref_driver.cc on arrays (uint64 arithmetic wraps)"""
    u = lambda v: np.asarray(v).astype(np.uint32).astype(np.uint64)
    with np.errstate(over="ignore"):
        x = (u(a) * np.uint64(0x9E3779B97F4A7C15)) ^ (u(b) * np.uint64(0xC2B2AE3D27D4EB4F)) ^ (u(c) * np.uint64(0x165667B19E3779F9)) \
            ^ (j.astype(np.uint64) * np.uint64(0xD6E8FEB86659FD93))
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return x


def _segmented_sum(x, off):
    """wrapping uint64 sums of x[off[k]:off[k+1]]"""
    n = len(off) - 1
    out = np.zeros(n, np.uint64)
    if len(x) == 0 or n == 0:
        return out
    with np.errstate(over="ignore"):
        cs = np.concatenate([np.zeros(1, np.uint64), np.cumsum(x, dtype=np.uint64)])
        out[:] = cs[off[1:]] - cs[off[:-1]]
    return out


def view_digests(res, n_bundles):
    """[NB, 3] uint64 from the views of agpu_batch_results(EVIDENCE | FRAGMENTS): the digests ref_timing_digest forms from the
    reference's own bundle objects (mmap segments, frgs, splices), per bundle"""
    ev, fr = res.evidence, res.fragments
    out = np.zeros((n_bundles, 3), np.uint64)
    for col, (off_p, val_p, width) in enumerate(((ev.seg_off, ev.seg, 3), (fr.frg_off, fr.frgs, 3), (ev.splice_off, ev.splices, 1))):
        off = np.ctypeslib.as_array(off_p, shape=(n_bundles + 1,)).astype(np.int64)
        tot = int(off[-1])
        if tot == 0:
            continue
        v = np.ctypeslib.as_array(val_p, shape=(tot * width,)).reshape(tot, width)
        j = np.arange(tot, dtype=np.int64) - np.repeat(off[:-1], np.diff(off))
        z = np.zeros(tot, np.int32)
        x = _mix_rows(v[:, 0], v[:, 1] if width > 1 else z, v[:, 2] if width > 2 else z, j)
        out[:, col] = _segmented_sum(x, off)
    return out


DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much
DUMP_SEED = 20260901        # seeds the choice of the bundles whose results are written
DUMP_HIT_BYTES = 256        # bound on the float64 result bytes per admitted hit of the sample; the log line shows the actual value


def _rows_index(off, rows, width=1):
    """element indices of rows `rows` of a ragged array whose row r holds elements [off[r] * width, off[r + 1] * width)"""
    s, n = off[rows] * width, (off[rows + 1] - off[rows]) * width
    return np.repeat(s - np.concatenate([[0], np.cumsum(n)[:-1]]).astype(np.int64), n) + np.arange(int(n.sum()), dtype=np.int64)


def result_arrays(res, nb, hit_off, rows):
    """the views of agpu_batch_results(ALL) (include/aletsch_gpu.h) restricted to the bundles `rows` of the batch, as float64
    arrays named <view>.<field>; a ragged field comes with <view>.<field>_len, its length per bundle (per cluster for the
    cluster and bridge fields)"""
    out = {}

    def view(ptr, n):
        return np.ctypeslib.as_array(ptr, shape=(int(n),)) if n > 0 else np.zeros(0)

    def ragged(name, ptr, off, sel, width=1):
        off = np.asarray(off, np.int64)
        out[name] = view(ptr, int(off[-1]) * width)[_rows_index(off, sel, width)]
        out[name + "_len"] = off[sel + 1] - off[sel]

    def fixed(name, ptr, n, sel, width=1):
        out[name] = view(ptr, n * width).reshape(-1, width)[sel].ravel() if n > 0 else np.zeros(0)

    def chainset(name, v, handle_off):
        bco = view(v.bundle_chain_off, nb + 1).astype(np.int64)
        ch = _rows_index(bco, rows)
        out[name + ".n_chains"] = bco[rows + 1] - bco[rows]
        ragged(name + ".chain_val", v.chain_val, view(v.chain_off, bco[-1] + 1), ch)
        fixed(name + ".chain_cnt", v.chain_cnt, bco[-1], ch, 3)
        fixed(name + ".chain_grp", v.chain_grp, bco[-1], ch)
        ragged(name + ".handle_chain", v.handle_chain, handle_off, rows)

    ev, fr, gr, cl, br = res.evidence, res.fragments, res.graph, res.clusters, res.bridges
    for f in ("lpos", "rpos", "strand"):
        fixed("evidence." + f, getattr(ev, f), nb, rows)
    ragged("evidence.seg", ev.seg, view(ev.seg_off, nb + 1), rows, 3)
    ragged("evidence.splices", ev.splices, view(ev.splice_off, nb + 1), rows)
    chainset("evidence.hcst", ev.hcst, hit_off)
    frg_off = view(fr.frg_off, nb + 1)
    ragged("fragments.frgs", fr.frgs, frg_off, rows, 3)
    chainset("fragments.fcst", fr.fcst, frg_off)
    fixed("fragments.bridged", fr.bridged, nb, rows)
    for f, width in (("junc", 9), ("pexon", 5), ("pexon_d", 4), ("vert", 5), ("vert_d", 3), ("edge", 3), ("edge_d", 1)):
        ragged("graph." + f, getattr(gr, f), view(getattr(gr, f.split("_")[0] + "_off"), nb + 1), rows, width)
    fixed("graph.strand", gr.strand, nb, rows)
    clu_off = view(cl.clu_off, nb + 1).astype(np.int64)
    nc = int(clu_off[-1])
    cs = _rows_index(clu_off, rows)
    out["clusters.n_clusters"] = clu_off[rows + 1] - clu_off[rows]
    for f, width in (("bounds", 4), ("extend", 4), ("count", 1), ("chain1", 1), ("chain2", 1)):
        fixed("clusters." + f, getattr(cl, f), nc, cs, width)
    ragged("clusters.frlist", cl.frlist, view(cl.frlist_off, nc + 1), cs)
    for f in ("type", "strand", "choices", "score"):
        fixed("bridges." + f, getattr(br, f), nc, cs)
    ragged("bridges.chain", br.chain, view(br.chain_off, nc + 1), cs)
    ragged("bridges.whole", br.whole, view(br.whole_off, nc + 1), cs)
    return {k: np.asarray(v, np.float64) for k, v in out.items()}


def dump_outputs(out_dir, bts, parts, per_bundle, counts):
    """--dump-outputs: what the timed path (reset + bridge_all) computed in its last step, as DIR/<name>.npy (float64): the
    batch counters, and bundle_counts plus every result view for a sample of bundles.  The sample depends on the input alone,
    so two builds dump the same bundles: the first bundles of a permutation drawn with DUMP_SEED whose admitted hits fit
    DUMP_BYTES at DUMP_HIT_BYTES each.  `bundle` holds the sampled bundles' indices."""
    from aletsch_b200 import gpu as G
    nb = sum(p.n_bundles for p in parts)
    order = np.random.default_rng(DUMP_SEED).permutation(nb)
    hits = np.concatenate([np.diff(p.a["bundle_hit_off"].astype(np.int64)) for p in parts])
    rows = np.sort(order[:int(np.searchsorted(np.cumsum(hits[order]), DUMP_BYTES // DUMP_HIT_BYTES, side="right"))])
    arrays = {"counts": np.array([counts[n] for n, _ in G.Counts._fields_], np.float64), "bundle": rows.astype(np.float64),
              "bundle_counts": np.asarray(per_bundle, np.float64)[rows].ravel()}
    first = 0
    per_part = []
    for x, part in zip(bts, parts):
        sel = rows[(rows >= first) & (rows < first + part.n_bundles)] - first
        first += part.n_bundles
        per_part.append(result_arrays(x.results(G.RESULT_ALL), part.n_bundles, part.a["bundle_hit_off"].astype(np.int64), sel))
    for name in per_part[0]:
        arrays[name] = np.concatenate([p[name] for p in per_part])
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit("bench.py --dump-outputs: the sampled results take %d bytes, more than %d; lower DUMP_BYTES / DUMP_HIT_BYTES"
                         % (total, DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("[bench] --dump-outputs: %d arrays, %.1f MB, %d of %d bundles, %.0f bytes per sampled hit -> %s" %
        (len(arrays), total / 1e6, len(rows), nb, total / max(1, int(hits[rows].sum())), out_dir))


def cpu_baseline(batch, cfg, threads, budget_s, gpu_bridged=None, gpu_digests=None):
    """the reference's own C++ (oracle/_ref) over a bounded sample of the same bundles (RefTimer), one untimed warm-up pass and
    then passes until the budget is used; the restatement (oracle/liboracle.so, kind "port") only if the reference build is absent"""
    if _checker_kind() != "reference":
        return cpu_baseline_port(batch, cfg, threads, budget_s, gpu_bridged)
    rt = RefTimer(batch, cfg, threads, max(2.0, budget_s / 3))
    rt.run()
    secs, bridged = [], 0
    t_end = time.time() + budget_s
    while not secs or (time.time() < t_end and len(secs) < 5):
        s_, bridged = rt.run()
        secs.append(s_)
    sec = float(np.mean(secs))
    out = {"value": rt.hits / sec, "unit": "hits/s", "cores": threads, "kind": "reference",
           "sample": rt.describe(sec), "passes": len(secs), "spread": float((max(secs) - min(secs)) / sec),
           "timed": "add_hit_intervals + build_fragments + bundle::bridge() per bundle (ref_timing_run); records and hit objects built before the clock, no dumps",
           "bridged_pairs_per_sec": bridged / sec}
    if gpu_bridged is not None:
        # full-size cross-check: the bridged-pair count of every sampled bundle, CUDA path vs this CPU run
        bad = [int(k) for k, c in zip(rt.sample, rt.per) if int(gpu_bridged[k]) != int(c)]
        out["bridged_count_check"] = {"bundles": len(rt.sample), "mismatches": len(bad), "first": bad[:5]}
    if gpu_digests is not None:
        # full-size cross-check of the arrays themselves: order-sensitive digests of every sampled bundle's mmap segments, frgs and
        # splices as the reference's own objects hold them after bundle::bridge() (untimed pass) vs the views the CUDA path returned
        want = rt.digests()
        got = gpu_digests[np.asarray(rt.sample, np.int64)] if len(rt.sample) else want
        bad = np.nonzero((want != got).any(axis=1))[0]
        out["array_digest_check"] = {"bundles": len(rt.sample), "arrays": ["mmap segments (l, r, cov)", "frgs (h1, h2, type)", "splices"],
                                     "mismatches": int(len(bad)), "first": [int(rt.sample[k]) for k in bad[:5]]}
    rt.close()
    return out


def cpu_baseline_port(batch, cfg, threads, budget_s, gpu_bridged=None):
    """fallback when oracle/_ref is absent: the CPU restatement through the checker interface (includes its result dumps)"""
    import orclib
    op = _orc_params(cfg)
    sizes = np.diff(batch.a["bundle_hit_off"])
    target_hits = int(60_000 * threads * budget_s)
    step = max(1, int(np.ceil(sizes.sum() / max(target_hits, 1))))
    sample = list(range(0, batch.n_bundles, step))
    bundles = [batch.bundle(k) for k in sample]
    hits = int(sum(len(b["pos"]) for b in bundles))
    lock = threading.Lock()
    nxt = [0]
    per = [0] * len(bundles)

    def worker():
        chk = orclib.Checker("orc")
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(bundles):
                return
            h = chk.new_bundle(bundles[i], op)
            chk.run_quiet(h, "fragments")
            per[i] = max(chk.run_quiet(h, "bridge"), 0)
            chk.free_bundle(h)

    t0 = time.time()
    ths = [threading.Thread(target=worker) for _ in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.time() - t0
    out = {"value": hits / dt, "unit": "hits/s", "cores": threads, "kind": "port",
           "sample": "every %d-th bundle of the same batch: %d bundles, %d hits, %.1f s wall" % (step, len(bundles), hits, dt),
           "bridged_pairs_per_sec": sum(per) / dt}
    if gpu_bridged is not None:
        bad = [int(k) for k, c in zip(sample, per) if int(gpu_bridged[k]) != int(c)]
        out["bridged_count_check"] = {"bundles": len(sample), "mismatches": len(bad), "first": bad[:5]}
    return out


def run_reference(args):
    """reference arm: the reference's own CPU implementation of the path on all host cores.  A step = one pass of
    ref_timing_run over a bounded sample of the workload's bundles sized for >= ~2 s of wall time; the sample is built once."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 8
    cfg = config_of(args)
    batch, n_records = build_workload(cfg, 0, ncpu)
    if _checker_kind() != "reference":
        r = cpu_baseline_port(batch, cfg, ncpu, max(2.0, args.cpu_seconds))
        vals, secs, hits_sample, kind, sample, bps = [r["value"]], [0.0], 0, "port", r["sample"], r["bridged_pairs_per_sec"]
    else:
        per_step = max(2.5, args.cpu_seconds / max(1, args.steps + args.warmup))
        rt = RefTimer(batch, cfg, ncpu, per_step)
        secs, br = [], 0
        for i in range(args.warmup + args.steps):
            s_, br = rt.run()
            if i >= args.warmup:
                secs.append(s_)
        hits_sample, kind = rt.hits, "reference"
        vals = [hits_sample / s_ for s_ in secs]
        sample = rt.describe(float(np.mean(secs)))
        bps = br / float(np.mean(secs))
        rt.close()
    value = float(np.mean(vals))
    config = reference_config(cfg, args, batch, n_records)
    out = {"metric": "hits_per_sec", "value": value, "unit": "hits/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * float(np.mean(secs)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
           "data": "synthetic", "impl": "reference", "config": config,
           "bridged_pairs_per_sec": bps,
           "ranks": "rank 0 only: one CPU pool of %d threads whatever N is (the GPU arm's value is the sum over N GPUs)" % ncpu,
           "spread": float((max(vals) - min(vals)) / value) if vals else 0.0,
           "cpu_baseline": {"value": value, "unit": "hits/s", "cores": ncpu, "kind": kind, "sample": sample,
                            "timed": "add_hit_intervals + build_fragments + bundle::bridge() per bundle; records and hit objects built before the clock, no dumps"},
           "e2e": {"value": value, "unit": "hits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_REAL_STDOUT = None


def quiet_stdout():
    """native libraries under us write to fd 1 (NCCL's version banner, the reference's statistics lines): send fd 1 to
    stderr for the whole run and keep the real stdout for the ONE JSON line"""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="index into BASELINE.json configs (default 1: the config the metric is quoted on)")
    ap.add_argument("--scale", type=float, default=None, help="fraction of the config's templates per sample (default: the config's own, 1.0 except configs[2])")
    ap.add_argument("--results", choices=["full", "bundle", "counts"], default="full",
                    help="what the end-to-end leg brings back to host memory per sub-batch (default: every result structure)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="CPU work budget of the bounded cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stage5", action="store_true", help="skip the bundle_group::resolve (stage 5) leg")
    ap.add_argument("--chunks", type=int, default=4, help="sub-batches of the end-to-end pipeline")
    ap.add_argument("--no-prefetch", action="store_true", help="end-to-end leg without the double-buffered asynchronous upload")
    ap.add_argument("--upload", choices=["compact", "lean"], default="compact",
                    help="host->device format of the end-to-end leg: agpu_batch_packed (default) or the lean agpu_batch_in")
    ap.add_argument("--streams", type=int, default=4, help="host threads / CUDA streams of the end-to-end pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
