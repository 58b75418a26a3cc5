"""The cross-sample cluster pass for a job that spans several device batches: the call a user makes when the bundles of all samples
do not fit one batch.

The cross-sample stages are bundle_group::resolve (stage 5, meta/bundle_group.cc:26-56), assembler::bridge (meta/assembler.cc:
977-1018, agpu_batch_group_bridge) and the support passes of assembler::assemble (meta/assembler.cc:177-373,
agpu_batch_group_support).  The two group calls take a cluster as bundle indices of ONE device batch, but the batching rule of the
ABI (include/aletsch_gpu.h, BATCHING RULE) cuts a large job by position into contiguous runs of bundles, while a stage-5 cluster
holds bundles of all samples at one locus.  So the job is cut twice, in the order assembler::resolve uses:

  1. by position (device_batches): evidence on every source batch, then every bundle's splice list (agpu_splices_fetch) -- all
     stage 5 needs;
  2. stage 5 over the region groups of the whole job (chromosome, 1 Mb region, strand: shard.bundle_region_keys);
  3. by cluster: every bundle of the job goes to exactly one output batch, laid out cluster by cluster (members in gv order), cut
     only at cluster boundaries under the same rule; the output batches are built on the device from the bundles already in HBM
     (agpu_batch_gather), then bridged per bundle, re-bridged per cluster and, if asked, given the support passes.

Evidence runs again on the output batches, on purpose: nothing derived (chain sets, coverage, ranks) is carried between batches.
Bundles are independent and a cluster's group pass depends only on its members in gv order, so every result equals the one of the
same job run as a single device batch.
"""
import time

import numpy as np

from . import gpu as G
from .shard import _cluster_pass

MAX_BATCH_SPAN = 3_000_000_000     # window positions per device batch: the coverage index is 32-bit (AGPU_ERR_CAPACITY above 2^32)
MAX_BATCH_HITS = 60_000_000


def bundle_spans(batch):
    """estimated coverage-window positions of every bundle of a host PackedBatch: [lpos, rpos) grown to 128-base alignment, where
    rpos may be a mate position up to 500 kb further (bundle_base::add_hit), with 512 positions of slack"""
    a = batch.a
    off = a["bundle_hit_off"]
    nb = batch.n_bundles
    if nb == 0:
        return np.zeros(0, np.int64)
    first = np.minimum(off[:-1], max(batch.n_hits - 1, 0))
    hi = np.maximum.reduceat(np.maximum(a["rpos"], np.where((a["mpos"] > a["rpos"]) & (a["mpos"] <= a["rpos"] + 500000), a["mpos"], 0)), first) \
        if batch.n_hits else np.zeros(nb, np.int64)
    return np.where(off[1:] > off[:-1], (hi.astype(np.int64) - a["pos"][first].astype(np.int64)) + 512, 256)


def _cuts(span, hits, unit=None):
    """greedy cut of a sequence of units (bundles or clusters) into runs with at most MAX_BATCH_SPAN window positions and
    MAX_BATCH_HITS hits, each run as long as the bounds allow.  A unit that alone exceeds a bound is a run of its own, or, when
    `unit` names it, a ValueError."""
    s = np.concatenate([[0], np.cumsum(np.asarray(span, np.int64))])
    h = np.concatenate([[0], np.cumsum(np.asarray(hits, np.int64))])
    n = len(span)
    cuts = [0]
    while cuts[-1] < n:
        c0 = cuts[-1]
        c1 = min(int(np.searchsorted(s, s[c0] + MAX_BATCH_SPAN, "right")), int(np.searchsorted(h, h[c0] + MAX_BATCH_HITS, "right"))) - 1
        if c1 <= c0:
            if unit is not None:
                raise ValueError("%s %d alone exceeds the batching rule (%d window positions, %d hits; at most %d and %d per device batch)"
                                 % (unit, c0, int(s[c0 + 1] - s[c0]), int(h[c0 + 1] - h[c0]), MAX_BATCH_SPAN, MAX_BATCH_HITS))
            c1 = c0 + 1
        cuts.append(c1)
    return cuts


def device_batches(batch):
    """The batching rule of the ABI: one device batch holds < 2^32 coverage-window positions (agpu_batch_evidence returns
    AGPU_ERR_CAPACITY otherwise).  Cuts a host PackedBatch into contiguous runs of whole bundles below MAX_BATCH_SPAN window positions
    and MAX_BATCH_HITS hits, with the window estimate of bundle_spans.  bench.py keeps a copy of the same rule; a later change can
    make it import this one."""
    if batch.n_bundles == 0:
        return [batch]
    cuts = _cuts(bundle_spans(batch), np.diff(batch.a["bundle_hit_off"]))
    if len(cuts) == 2:
        return [batch]
    return [batch.slice(cuts[i], cuts[i + 1]) for i in range(len(cuts) - 1)]


class ClusterPass:
    """What cluster_pass leaves, per output batch i:
      batches[i]   the gathered gpu.Batch, bridged per bundle and re-bridged per cluster (its fetch calls give the results)
      clusters[i]  its clusters of >= 2 bundles as lists of batch-local bundle indices in gv order (what group_bridge ran on)
      origin[i]    int64 [NB, 3]: per local bundle, the source part, the bundle index in that part and the bundle index in the job
      support[i]   the support rows of its clusters (gpu.Batch.group_support's dicts), when asked for; else None
      phases[i]    the combined phase set px of each of its clusters (gpu.Batch.group_phase_set's dicts), when asked for; else None
    and n_groups / n_clusters, the region-group and stage-5 cluster counts of the job, singletons included."""

    def __init__(self):
        self.batches, self.clusters, self.origin, self.support, self.phases = [], [], [], None, None
        self.n_groups = self.n_clusters = 0

    def free(self):
        for b in self.batches:
            b.free()
        self.batches = []


def _group_support(bt, clusters, params):
    """group_support, halving the cluster list while the (edge x sample) scratch of one call exceeds its bound"""
    try:
        return bt.group_support(clusters, params)
    except G.AgpuError as e:
        if e.rc != G.AGPU_ERR_CAPACITY or len(clusters) < 2:
            raise
    h = len(clusters) // 2
    return _group_support(bt, clusters[:h], params) + _group_support(bt, clusters[h:], params)


def cluster_pass(ctx, parts, batches, params, support=False, times=None, phases=False):
    """Stage 5, assembler::bridge, (support=True) the support passes and (phases=True) the clusters' combined phase sets over a
    job cut into several device batches.

    parts:   the host sub-batches (hostlib.PackedBatch): contiguous slices, in order, of one job, as device_batches returns them
    batches: the matching device batches (gpu.Batch, on any context of ctx's device), fresh: just uploaded or reset
    params:  gpu.Params, including max_group_size / min_grouping_similarity of stage 5
    times:   optional dict; receives host-clock seconds of every phase around synchronised work ('evidence', 'signatures', 'stage5',
             'plan', 'exchange', 'gather', and per output batch lists 'bridge_all', 'group_bridge', 'group_support', 'phase_set')
    The output batches live on ctx.  The caller owns the sources and may free them once this returns.  This is the sharded pass
    of one rank (shard.cluster_pass_sharded) with keys sample << 32 | job index, so nothing is communicated even when a process
    group exists."""
    sample = np.concatenate([p.a["bundle_sample"] for p in parts]).astype(np.int64) if parts else np.zeros(0, np.int64)
    keys = (sample << 32) | np.arange(len(sample), dtype=np.int64)
    out = _cluster_pass(ctx, parts, batches, keys, params, support, times, 0, 1, phases)
    out.origin = [np.stack([o[:, 2], o[:, 3], o[:, 1] & 0xffffffff], axis=1) for o in out.origin]
    return out


def run_clusters(ctx, sources, picks, span, hits, cstart, params, out, clock, support, origin, phases=False):
    """steps 3 and 4 of the pass on bundles laid out cluster by cluster: bundle k of the layout is bundle picks[k][1] of
    sources[picks[k][0]], with window estimate span[k] and hits[k]; cluster j is the layout range [cstart[j], cstart[j + 1]).
    Cuts the layout at cluster boundaries under the batching rule (ValueError for a cluster larger than one device batch), then
    per output batch: gather, bundle::bridge, assembler::bridge on its clusters, the support passes, and the members' phase sets
    against graphs rebuilt from the updated evidence with every cluster's combined phase set (a cluster lives in one output
    batch, so this needs nothing from other batches or ranks).  Appends to `out` (a ClusterPass), with origin[k] as the origin
    row of bundle k."""
    cuts = _cuts(np.add.reduceat(span, cstart[:-1]), np.add.reduceat(hits, cstart[:-1]), unit="cluster") if len(cstart) > 1 else [0]
    clock.lap("plan", add=True)
    for k0, k1 in zip(cuts[:-1], cuts[1:]):
        b0, b1 = int(cstart[k0]), int(cstart[k1])
        bt = ctx.gather(sources, picks[b0:b1])
        out.batches.append(bt)
        out.origin.append(origin[b0:b1])
        clock.lap("gather", add=True)
        bt.bridge_all(params)
        clock.lap("bridge_all", per_batch=True)
        multi = [list(range(int(cstart[k]) - b0, int(cstart[k + 1]) - b0)) for k in range(k0, k1) if cstart[k + 1] - cstart[k] >= 2]
        out.clusters.append(multi)
        if multi:
            bt.group_bridge(multi, params)
        clock.lap("group_bridge", per_batch=True)
        if support:
            out.support.append(_group_support(bt, multi, params) if multi else [])
            clock.lap("group_support", per_batch=True)
        if phases:
            if multi:
                bt.graph(params)
                bt._run("phase_set")
            out.phases.append(bt.group_phase_set(multi) if multi else [])
            clock.lap("phase_set", per_batch=True)


class _Clock:
    """host clock around synchronised work, when the caller asked for phase times"""

    def __init__(self, ctx, batches, times):
        self.ctxs = [ctx] + [b.ctx for b in batches if b.ctx is not ctx]
        self.times = times
        self.t = time.perf_counter() if times is not None else 0.0

    def lap(self, name, add=False, per_batch=False):
        if self.times is None:
            return
        for c in self.ctxs:
            c.sync()
        now = time.perf_counter()
        dt, self.t = now - self.t, now
        if per_batch:
            self.times.setdefault(name, []).append(dt)
        else:
            self.times[name] = self.times.get(name, 0.0) + dt if add else dt
