"""Multi-GPU plumbing of the path (SURVEY.md section 8e): one process per GPU, torch.distributed.

Stages 1-4 are per bundle and need no collective: work units (regions, i.e. all bundles of one
(chromosome, 1 Mb region) key, meta/incubator.cc:357-381) are dealt to ranks by longest-processing-
time-first on their hit counts.  The only exchange of the path is for stage 5 when samples are
ingested on different ranks: the per-bundle splice lists (bundle::splices, the "junction
signatures") of a region group are all-gathered so that every rank runs the identical
bundle_group::resolve (meta/bundle_group.cc:26-56) and learns which bundles it has to receive.

cluster_pass_sharded builds the rest of the cross-sample pass on that: the same all-gather also carries every bundle's hits, CIGAR
operations and window estimate, every rank computes the same plan (plan_clusters: which rank owns which cluster, single-bundle
clusters staying where they were ingested), the bundles of every cluster move to its owner (one device gather per peer, the
batch's device columns sent with NCCL point-to-point, adopted on the receiving side without a copy), and the owner runs
assembler::bridge and the support passes on its clusters (clusters.run_clusters).  With one rank the same pass runs without any
communication: that is clusters.cluster_pass.
Backend: NCCL over NVLink on GPUs; the CPU tests run the same code over gloo.
"""
import numpy as np
import torch
import torch.distributed as dist


def assign_units(weights, world, load=None):
    """LPT: units (descending weight, ties by index) go to the currently lightest rank (ties by rank).  `load`: optional initial
    load of every rank (work it holds already).  Returns rank_of[unit]; deterministic, identical on every rank."""
    w = np.asarray(weights, np.int64)
    order = sorted(range(len(w)), key=lambda i: (-int(w[i]), i))
    load = [0] * world if load is None else [int(x) for x in load]
    rank_of = np.zeros(len(w), np.int32)
    for i in order:
        r = min(range(world), key=lambda k: (load[k], k))
        rank_of[i] = r
        load[r] += int(w[i])
    return rank_of


def _device():
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


REGION = 1_000_000      # region_partition_length (util/parameters.cc:42)


def gather_packed(off, val, keys, extra=None):
    """all-gather of packed variable-length int32 lists (vectorised: no per-list Python work).

    off[n+1] / val: this rank's lists; keys[n] (int64) and extra (int64, optional: [n], or [n, m] for m columns) travel with them.
    Two collectives: the per-rank (n_lists, n_values) header, then one padded int64 payload [lengths | keys | extra columns |
    values].  Returns (off_all, val_all, keys_all, extra_all, owner_rank) concatenated in rank order, identical on every rank, with
    extra_all shaped like extra, plus the bytes this rank received."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    off = np.asarray(off, np.int64)
    val = np.asarray(val, np.int32)
    n = len(off) - 1
    keys = np.asarray(keys, np.int64)
    extra = np.zeros(n, np.int64) if extra is None else np.asarray(extra, np.int64)
    m = 1 if extra.ndim == 1 else extra.shape[1]
    lens = np.diff(off)
    if world == 1:
        return off, val, keys, extra, np.zeros(n, np.int32), 0
    dev = _device()
    head = torch.tensor([n, int(lens.sum())], dtype=torch.int64, device=dev)
    heads = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(heads, head)
    heads = [h.cpu().numpy() for h in heads]
    cap = max(int((2 + m) * h[0] + h[1]) for h in heads)
    payload = np.concatenate([lens, keys, extra.T.reshape(-1), val.astype(np.int64)])
    mine = torch.zeros(max(cap, 1), dtype=torch.int64, device=dev)
    if len(payload):
        mine[:len(payload)] = torch.from_numpy(payload).to(dev)
    parts = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    lens_all, keys_all, extra_all, vals_all, owner = [], [], [], [], []
    for r in range(world):
        nr, nv = int(heads[r][0]), int(heads[r][1])
        p = parts[r].cpu().numpy()
        lens_all.append(p[:nr]); keys_all.append(p[nr:2 * nr])
        x = p[2 * nr:(2 + m) * nr]
        extra_all.append(x if extra.ndim == 1 else x.reshape(m, nr).T)
        vals_all.append(p[(2 + m) * nr:(2 + m) * nr + nv].astype(np.int32))
        owner.append(np.full(nr, r, np.int32))
    lens_all = np.concatenate(lens_all)
    off_all = np.zeros(len(lens_all) + 1, np.int64)
    np.cumsum(lens_all, out=off_all[1:])
    return off_all, np.concatenate(vals_all), np.concatenate(keys_all), np.concatenate(extra_all), np.concatenate(owner), int(8 * cap * world)


def resolve_region_groups(ctx, off, val, keys, region_key, params):
    """bundle_group::resolve for a job whose SAMPLES are ingested on different ranks (meta/incubator.cc:461-471: a bundle group
    holds the bundles of ALL samples of one (chromosome, region, strand)).  Every rank contributes the splice signatures of its
    own bundles with their global keys (e.g. sample << 32 | bundle-in-sample) and region keys; after ONE all-gather every rank
    orders the bundles canonically -- (region key, key): the gset order must not depend on the rank count -- and runs the
    identical agpu_group_resolve_batch on its own GPU.  Returns (keys_sorted, region_sorted, cluster_of, owner_sorted,
    bytes_received): cluster_of[i] is the cluster of bundle keys_sorted[i] inside its region group."""
    off_all, val_all, keys_all, reg_all, owner, nbytes = gather_packed(off, val, keys, region_key)
    order, cl_of = _resolve_sorted(ctx, off_all, val_all, keys_all, reg_all, params)
    return keys_all[order], reg_all[order], cl_of, owner[order], nbytes


def _resolve_sorted(ctx, off_all, val_all, keys_all, reg_all, params):
    """stage 5 over gathered signatures: the canonical (region key, key) order and the cluster of every bundle in that order"""
    from . import gpu as G
    order = np.lexsort((keys_all, reg_all))
    loff, lval = G.reorder_lists(off_all, val_all, order)
    reg_s = reg_all[order]
    cuts = np.concatenate([[0], np.nonzero(np.diff(reg_s))[0] + 1, [len(reg_s)]]) if len(reg_s) else np.zeros(1, np.int64)
    group_off = np.asarray(cuts, np.int32)
    cl_of, _ = G.group_resolve_arrays(ctx, group_off, loff, lval, params)
    return order, cl_of[:len(order)]


def bundle_region_keys(batch):
    """(chromosome, 1 Mb region, strand) key of every bundle of a packed host batch; for unstranded libraries the strand is the
    majority of the hits' XS tags (bundle_base::compute_strand, rnacore/bundle_base.cc:206-224)"""
    a = batch.a
    off = a["bundle_hit_off"]
    if batch.n_bundles == 0:
        return np.zeros(0, np.int64)
    first = np.minimum(off[:-1], max(batch.n_hits - 1, 0))
    strand = a["strand"][first].astype(np.int64)
    if batch.n_hits and np.any(strand == ord(".")):
        cp = np.concatenate([[0], np.cumsum(a["xs"] == ord("+"))])
        cm = np.concatenate([[0], np.cumsum(a["xs"] == ord("-"))])
        npl, nmi = cp[off[1:]] - cp[off[:-1]], cm[off[1:]] - cm[off[:-1]]
        strand = np.where(strand == ord("."), np.where(npl > nmi, ord("+"), np.where(npl < nmi, ord("-"), ord("."))), strand)
    return (a["bundle_tid"].astype(np.int64) << 40) | ((a["pos"][first].astype(np.int64) // REGION) << 8) | strand


# ---- the cross-sample cluster pass with samples ingested on different ranks ---------------------------------------------------

class Plan:
    """Who owns which stage-5 cluster (plan_clusters), the same on every rank:
      rows[r]    indices into the planner's input arrays of the bundles rank r lays out, in its layout order
      cstart[r]  cluster starts in rows[r] (len = its clusters + 1)
      dest       owner rank of every cluster of the job, clusters in global layout order
      size       member count of every cluster; load[r] hits rank r owns"""

    def __init__(self, rows, cstart, dest, size, load):
        self.rows, self.cstart, self.dest, self.size, self.load = rows, cstart, dest, size, load

    @property
    def n_clusters(self):
        return len(self.dest)


def plan_clusters(keys, region, cluster, owner, hits, span, world):
    """Deal the stage-5 clusters of a job to ranks; no communication.  Per bundle of the whole job, in any order: its key
    (sample << 32 | index in its sample), region key, cluster inside its region group, ingesting rank, hits and coverage-window
    estimate (clusters.bundle_spans).  A cluster is a (region group, cluster) pair with its members in (region key, key) order --
    for such keys the gv order (region, sample, job index) cluster_pass uses.  A single-bundle cluster stays on its ingesting
    rank; clusters of several bundles go by LPT on their hits, each rank's load seeded with its singletons' hits.  Every owner
    lays out its clusters in the global layout order (region groups in order, clusters in gvv order, members in gv order); a
    cluster larger than one device batch raises the ValueError of clusters._cuts on every rank."""
    from .clusters import _cuts
    keys, region, cluster = np.asarray(keys, np.int64), np.asarray(region, np.int64), np.asarray(cluster, np.int64)
    owner, hits, span = np.asarray(owner, np.int64), np.asarray(hits, np.int64), np.asarray(span, np.int64)
    n = len(keys)
    lay = np.lexsort((keys, cluster, region))
    new = (np.diff(region[lay]) != 0) | (np.diff(cluster[lay]) != 0)
    cstart = np.concatenate([[0], np.nonzero(new)[0] + 1, [n]]).astype(np.int64) if n else np.zeros(1, np.int64)
    size = np.diff(cstart)
    chits = np.add.reduceat(hits[lay], cstart[:-1]) if n else np.zeros(0, np.int64)
    dest = owner[lay[cstart[:-1]]].copy()
    one = size == 1
    seed = np.bincount(dest[one], weights=chits[one], minlength=world).astype(np.int64)
    dest[~one] = assign_units(chits[~one], world, seed)
    rows, starts = [], []
    for r in range(world):
        cl = np.nonzero(dest == r)[0]
        st = np.concatenate([[0], np.cumsum(size[cl])]).astype(np.int64)
        idx = np.repeat(cstart[cl] - st[:-1], size[cl]) + np.arange(int(st[-1]), dtype=np.int64)
        rows.append(lay[idx])
        starts.append(st)
        if len(cl):
            _cuts(np.add.reduceat(span[lay[idx]], st[:-1]), np.add.reduceat(hits[lay[idx]], st[:-1]), unit="cluster")
    load = np.bincount(dest, weights=chits, minlength=world).astype(np.int64)
    return Plan(rows, starts, dest, size, load)


def bundle_keys(batch):
    """global key of every bundle of a host batch: sample << 32 | index of the bundle among its sample's bundles"""
    sample = batch.a["bundle_sample"].astype(np.int64)
    order = np.argsort(sample, kind="stable")
    within = np.empty(len(sample), np.int64)
    within[order] = np.arange(len(sample)) - np.searchsorted(sample[order], sample[order])
    return (sample << 32) | within


# the hit and CIGAR columns of a batch that travel between ranks (gpu.Batch.input_columns); bundle_hit_off, bundle_tid and
# bundle_sample are rebuilt from the plan on the receiving side
SENT_COLUMNS = (("pos", torch.int32), ("rpos", torch.int32), ("mpos", torch.int32), ("isize", torch.int32), ("strand", torch.int8),
                ("xs", torch.int8), ("qid", torch.int64), ("cigar_off", torch.int32), ("cigar", torch.int32))


def _exchange(ctx, batches, base, plan, g, rank, world, stats):
    """Move the bundles of the clusters this rank owns from their ingesting ranks: per peer one agpu_batch_gather of what it
    needs (in its layout order), all columns of all peers in one batch_isend_irecv, received into torch tensors and adopted as
    one batch per peer.  g: the gathered per-bundle arrays (keys, region, owner, local index, hits, ops).  Returns
    {peer: adopted gpu.Batch}."""
    dev = _device()
    ops, sends, recv = [], [], {}
    for d in range(world):
        if d == rank:
            continue
        out = plan.rows[d][g["owner"][plan.rows[d]] == rank]
        if len(out):
            li = g["local"][out]
            part = np.searchsorted(base, li, "right") - 1
            bt = ctx.gather(batches, np.stack([part, li - base[part]], axis=1))
            cols = bt.input_columns()
            sends.append(bt)
            for tag, (name, _) in enumerate(SENT_COLUMNS):
                t = cols[name]
                if t.numel():
                    ops.append(dist.P2POp(dist.isend, t, d, tag=tag))
                    stats["bytes_sent"] += t.numel() * t.element_size()
                    stats["bytes_to"][d] += t.numel() * t.element_size()
            stats["bundles_sent"] += len(out)
            stats["hits_sent"] += int(g["hits"][out].sum())
        inn = plan.rows[rank][g["owner"][plan.rows[rank]] == d]
        if len(inn):
            nh, nc = int(g["hits"][inn].sum()), int(g["ops"][inn].sum())
            size = {"cigar_off": nh + 1, "cigar": nc}
            bufs = {}
            for tag, (name, dt) in enumerate(SENT_COLUMNS):
                m = size.get(name, nh)
                bufs[name] = torch.empty(max(m, 1), dtype=dt, device=dev)
                if m:
                    ops.append(dist.P2POp(dist.irecv, bufs[name][:m], d, tag=tag))
                    stats["bytes_received"] += m * bufs[name].element_size()
                    stats["bytes_from"][d] += m * bufs[name].element_size()
            hit_off = np.concatenate([[0], np.cumsum(g["hits"][inn])]).astype(np.int64)
            bufs["bundle_hit_off"] = torch.from_numpy(hit_off).to(dev)
            bufs["bundle_tid"] = torch.from_numpy((g["region"][inn] >> 40).astype(np.int32)).to(dev)
            bufs["bundle_sample"] = torch.from_numpy((g["keys"][inn] >> 32).astype(np.int32)).to(dev)
            recv[d] = (bufs, len(inn), nh, nc)
            stats["bundles_received"] += len(inn)
            stats["hits_received"] += nh
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    if dev.type == "cuda":
        torch.cuda.current_stream(dev).synchronize()     # the library's stream does not see NCCL's
    for bt in sends:
        bt.free()
    from . import hostlib as H
    adopted = {}
    for d, (bufs, nb, nh, nc) in recv.items():
        b = H.BatchIn()
        b.n_bundles, b.n_hits, b.n_cigar = nb, nh, nc
        for name in ("bundle_hit_off", "bundle_tid", "bundle_sample") + tuple(n for n, _ in SENT_COLUMNS):
            setattr(b, name, bufs[name].data_ptr())
        adopted[d] = ctx.adopt(b, keepalive=bufs)
    return adopted


def cluster_pass_sharded(ctx, parts, batches, keys, params, support=False, times=None, phases=False):
    """clusters.cluster_pass for a job whose samples are ingested on different ranks (one process per GPU).

    parts / batches: this rank's host parts and device batches, as cluster_pass takes them; keys: the global key of every bundle
    of the parts, in order (sample << 32 | index of the bundle in its sample).  Evidence and the splice lists run on the sources;
    one all-gather carries every bundle's signature, region key, hits, CIGAR operations and window estimate; every rank runs the
    same stage 5 and the same plan (plan_clusters); the members of every cluster this rank owns that were ingested elsewhere are
    moved here (NCCL point-to-point between the GPUs, nothing staged through host memory; gloo on the CPU tier); then steps 3
    and 4 of cluster_pass (clusters.run_clusters) run on this rank's clusters.

    Returns a clusters.ClusterPass for this rank's clusters; its origin rows are (ingesting rank, global key, local part, index in
    the part), the last two -1 for a bundle received from another rank, and n_groups / n_clusters count the region groups and
    clusters of the whole job.  `.exchange` holds the bundles, hits and bytes this rank sent and received, and the bytes per peer
    (bytes_to, bytes_from).  times: cluster_pass's phase times; phases: cluster_pass's combined phase sets, of this rank's
    clusters.  Without a process group the result equals cluster_pass's."""
    grouped = dist.is_available() and dist.is_initialized()
    rank, world = (dist.get_rank(), dist.get_world_size()) if grouped else (0, 1)
    return _cluster_pass(ctx, parts, batches, keys, params, support, times, rank, world, phases)


def _cluster_pass(ctx, parts, batches, keys, params, support, times, rank, world, phases=False):
    """the cross-sample cluster pass as rank `rank` of `world`; with world 1 nothing is communicated, whatever process group exists"""
    from .clusters import ClusterPass, _Clock, bundle_spans, run_clusters
    if len(parts) != len(batches):
        raise ValueError("cluster pass: %d host parts but %d device batches" % (len(parts), len(batches)))
    keys = np.asarray(keys, np.int64)
    base = np.concatenate([[0], np.cumsum([p.n_bundles for p in parts])]).astype(np.int64)
    if len(keys) != base[-1]:
        raise ValueError("cluster pass: %d keys for %d bundles" % (len(keys), base[-1]))
    clock = _Clock(ctx, batches, times)
    out = ClusterPass()
    out.support = [] if support else None
    out.phases = [] if phases else None
    out.exchange = {k: 0 for k in ("bundles_sent", "hits_sent", "bytes_sent", "bundles_received", "hits_received", "bytes_received")}
    out.exchange.update(bytes_to=[0] * world, bytes_from=[0] * world)
    # 1. evidence on the sources, then bundle::splices of this rank's bundles
    offs, vals, vb = [np.zeros(1, np.int64)], [], 0
    for bt in batches:
        bt.evidence(params)
        o, v = bt.fetch_splices()
        offs.append(o[1:] + vb)
        vals.append(v)
        vb += int(o[-1])
    off, val = np.concatenate(offs), np.concatenate(vals) if vals else np.zeros(0, np.int32)
    clock.lap("evidence")
    # 2. one all-gather: signatures with (region key, hits, CIGAR operations, window estimate) per bundle; stage 5 on every rank
    cols = np.zeros((len(keys), 4), np.int64)
    if len(keys):
        hit_off = [p.a["bundle_hit_off"] for p in parts]
        cols[:, 0] = np.concatenate([bundle_region_keys(p) for p in parts])
        cols[:, 1] = np.concatenate([np.diff(h) for h in hit_off])
        cols[:, 2] = np.concatenate([np.diff(p.a["cigar_off"][h].astype(np.int64)) for p, h in zip(parts, hit_off)])
        cols[:, 3] = np.concatenate([bundle_spans(p) for p in parts])
    if world > 1:
        off_all, val_all, keys_all, x, owner, _ = gather_packed(off, val, keys, cols)
    else:
        off_all, val_all, keys_all, x, owner = off, val, keys, cols, np.zeros(len(keys), np.int32)
    clock.lap("signatures")
    n = len(keys_all)
    if n == 0:
        return out
    order, cl_sorted = _resolve_sorted(ctx, off_all, val_all, keys_all, x[:, 0], params)
    cl_of = np.empty(n, np.int64)
    cl_of[order] = cl_sorted
    out.n_groups = 1 + int(np.count_nonzero(np.diff(x[order, 0])))
    clock.lap("stage5")
    # 3. the plan, the same on every rank
    plan = plan_clusters(keys_all, x[:, 0], cl_of, owner, x[:, 1], x[:, 3], world)
    first = np.searchsorted(owner, np.arange(world))          # gather_packed concatenates in rank order
    g = {"keys": keys_all, "region": x[:, 0], "owner": owner, "local": np.arange(n) - first[owner], "hits": x[:, 1], "ops": x[:, 2]}
    out.n_clusters = plan.n_clusters
    out.load = plan.load
    clock.lap("plan")
    adopted = _exchange(ctx, batches, base, plan, g, rank, world, out.exchange) if world > 1 else {}
    clock.lap("exchange")
    # 4. the layout of this rank's clusters: local bundles from the sources, the others from the batch of their peer
    rows = plan.rows[rank]
    src_of = owner[rows]
    local = src_of == rank
    li = g["local"][rows]
    part = np.where(local, np.searchsorted(base, li, "right") - 1, -1)
    idx = np.where(local, li - base[np.maximum(part, 0)], -1)
    peers = sorted(adopted)
    picks = np.stack([part, idx], axis=1)
    for k, d in enumerate(peers):
        m = src_of == d
        picks[m, 0] = len(batches) + k
        picks[m, 1] = np.arange(int(m.sum()))
    origin = np.stack([src_of, keys_all[rows], part, idx], axis=1).astype(np.int64)
    try:
        run_clusters(ctx, list(batches) + [adopted[d] for d in peers], picks, x[rows, 3], x[rows, 1], plan.cstart[rank], params, out,
                     clock, support, origin, phases)
    finally:
        for b in adopted.values():
            b.free()
    return out
