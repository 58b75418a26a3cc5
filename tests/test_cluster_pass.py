"""agpu_batch_gather (bundles regrouped on the device) and the cluster pass over a job cut into several device batches
(aletsch_b200/clusters.py).  The oracle is the single-batch device path, which the parity tests pin to the CPU checkers: bundles
are independent, and a cluster's group pass depends only on its members in gv order.  CPU tier: kernel-logic build; -m gpu: the
CUDA path."""
import numpy as np
import pytest

import bench
import fuzz
import parity
from aletsch_b200 import clusters as CL
from aletsch_b200 import gpu as G
from aletsch_b200 import hostlib as H


def all_results(bt, nb, hit_off, rows=None):
    """every view of agpu_batch_results(ALL) for the bundles `rows` (all by default), as named arrays"""
    rows = np.arange(nb) if rows is None else np.asarray(rows, np.int64)
    return bench.result_arrays(bt.results(G.RESULT_ALL), nb, np.asarray(hit_off, np.int64), rows)


def diff_arrays(a, b, where):
    if sorted(a) != sorted(b):
        return ["%s: names differ: %s vs %s" % (where, sorted(a), sorted(b))]
    return ["%s: %s differs" % (where, k) for k in sorted(a) if a[k].shape != b[k].shape or not np.array_equal(a[k], b[k])]


def upload_three_ways(ctxs, parts):
    """part 0 with every array, part 1 lean (no rpos, bundle_strand only), part 2 in the compact form"""
    c = [ctxs[k % len(ctxs)] for k in range(3)]
    arr = parts[2].compact()
    return [c[0].upload(parts[0].view(), keepalive=parts[0]), c[1].upload(parity.lean_view(parts[1]), keepalive=parts[1]),
            c[2].upload(H.compact_struct(arr, parts[2].n_cigar), keepalive=(arr, parts[2]))]


def picks_of(parts, glob):
    base = np.concatenate([[0], np.cumsum([p.n_bundles for p in parts])])
    part = np.searchsorted(base, glob, "right") - 1
    return np.stack([part, glob - base[part]], axis=1)


def check_gather(lib, batch, lt, free_sources=False, other_contexts=False, seed=7):
    ctx = G.Context(0, lib_path=lib)
    others = [G.Context(0, lib_path=lib), G.Context(0, lib_path=lib)] if other_contexts else [ctx]
    gp = G.default_params(library_type=lt)
    parts = batch.split(3)
    assert len(parts) == 3
    srcs = upload_three_ways(others, parts)
    rng = np.random.default_rng(seed)
    glob = rng.permutation(batch.n_bundles)
    glob = np.concatenate([glob, rng.choice(glob, 5)])             # a few bundles twice
    picks = picks_of(parts, glob)
    assert len(set(picks[:50, 0].tolist())) == 3
    gb = ctx.gather(srcs, picks)
    if free_sources:
        for s in srcs:
            s.free()
    sel = batch.select(glob)
    ref = ctx.upload(sel.view(), keepalive=sel)
    gb.bridge_all(gp)
    ref.bridge_all(gp)
    assert gb.counts() == ref.counts()
    assert np.array_equal(gb.bundle_counts(), ref.bundle_counts())
    want = all_results(ref, sel.n_bundles, sel.a["bundle_hit_off"])
    got = all_results(gb, sel.n_bundles, sel.a["bundle_hit_off"])
    bad = diff_arrays(want, got, "gather vs select")
    assert not bad, bad[:5]
    stats = {"bundles": len(glob), "hits": int(sel.n_hits), "bridged": gb.counts()["bridged"]}
    for b in [gb, ref] + srcs:
        b.free()
    for c in set(others + [ctx]):
        c.close()
    return stats


def check_edges(lib):
    ctx = G.Context(0, lib_path=lib)
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 8000, samples=2)
    gp = G.default_params(library_type=lt)
    parts = batch.split(2)
    srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
    # nothing selected: a valid empty batch
    e = ctx.gather(srcs, np.zeros((0, 2), np.int32))
    e.bridge_all(gp)
    c = e.counts()
    assert c["hits"] == 0 and c["cigar_ops"] == 0 and c["fragments"] == 0
    e.free()
    # indices out of range
    for bad in ([(0, parts[0].n_bundles)], [(2, 0)], [(-1, 0)], [(1, -1)]):
        with pytest.raises(G.AgpuError) as ex:
            ctx.gather(srcs, bad)
        assert ex.value.rc == G.AGPU_ERR_ARG
    # a source with coverage edits
    ed = ctx.upload(parts[1].view(), keepalive=parts[1])
    ed.coverage_edit(skip=np.zeros(parts[1].n_hits, np.uint16))
    with pytest.raises(G.AgpuError) as ex:
        ctx.gather([srcs[0], ed], [(0, 0), (1, 0)])
    assert ex.value.rc == G.AGPU_ERR_ARG
    ed.free()
    # the context still works
    g = ctx.gather(srcs, [(1, 0), (0, 1), (1, 0)])
    g.bridge_all(gp)
    assert g.counts()["hits"] > 0
    g.free()
    for s in srcs:
        s.free()
    # a packing-contract violation in one bundle surfaces at the output's evidence exactly when that bundle is selected
    fz = fuzz.random_batch(11, n_bundles=8, max_hits=40)
    off = fz.a["bundle_hit_off"]
    k = int(np.nonzero(np.diff(off) >= 2)[0][0])
    fz.a["pos"][off[k] + 1] = fz.a["pos"][off[k]] - 3                # hits out of order
    src = ctx.upload(fz.view(), keepalive=fz)
    fp = G.default_params(library_type=H.FR_FIRST)
    for chosen in ([j for j in range(8) if j != k], [k], list(range(8))):
        g = ctx.gather([src], [(0, j) for j in chosen])
        if k in chosen:
            with pytest.raises(G.AgpuError) as ex:
                g.evidence(fp)
            assert ex.value.rc == G.AGPU_ERR_INPUT
        else:
            g.evidence(fp)
        g.free()
    src.free()
    ctx.close()


def single_batch_run(ctx, batch, gp):
    """the oracle: the whole job as one device batch -- bridge_all, stage 5 over the region groups, group_bridge, group_support"""
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
    bt.group_bridge(multi, gp)
    rows = bt.group_support(multi, gp)
    return bt, multi, bt.fetch_group(), rows


def check_cluster_pass(lib, mode, templates, samples, monkeypatch):
    ctx1, ctx2 = G.Context(0, lib_path=lib), G.Context(0, lib_path=lib)
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    whole, multi, cb_want, sup_want = single_batch_run(ctx1, batch, gp)
    assert len(multi) >= 5
    per_bundle_want = whole.bundle_counts()
    parts = batch.split(3)
    srcs = [ctx2.upload(p.view(), keepalive=p) for p in parts]
    # output batches of about a third of the job each: the cut by cluster is exercised too
    monkeypatch.setattr(CL, "MAX_BATCH_HITS", batch.n_hits // 3 + 1)
    res = CL.cluster_pass(ctx2, parts, srcs, gp, support=True)
    for s in srcs:
        s.free()
    # every bundle in exactly one output batch; clusters identical, in the same order
    glob = np.concatenate([o[:, 2] for o in res.origin])
    assert np.array_equal(np.sort(glob), np.arange(batch.n_bundles))
    got_multi = [[int(o[m, 2]) for m in c] for o, cl in zip(res.origin, res.clusters) for c in cl]
    assert got_multi == multi
    spanning = sum(len(set(o[c, 0].tolist())) > 1 for o, cl in zip(res.origin, res.clusters) for c in cl)
    assert spanning > 0, "no cluster spans the parts: the cut tests nothing"
    bad = []
    hit_off = batch.a["bundle_hit_off"]
    nh = np.diff(hit_off)
    for i, (bt, o) in enumerate(zip(res.batches, res.origin)):
        want = all_results(whole, batch.n_bundles, hit_off, o[:, 2])
        loc_off = np.concatenate([[0], np.cumsum(nh[o[:, 2]])])
        bad += diff_arrays(want, all_results(bt, len(o), loc_off), "output batch %d" % i)
        if not np.array_equal(bt.bundle_counts(), per_bundle_want[o[:, 2]]):
            bad.append("output batch %d: bundle_counts differ" % i)
    cb_got = [d for bt, cl in zip(res.batches, res.clusters) if cl for d in bt.fetch_group()]
    sup_got = [d for s in res.support for d in s]
    assert len(cb_got) == len(cb_want) == len(sup_got) == len(sup_want)
    for gi in range(len(multi)):
        bad += diff_arrays(cb_want[gi], cb_got[gi], "cluster %d combined bundle" % gi)
        w, g = sup_want[gi], sup_got[gi]
        if sorted(w) != sorted(g):
            bad.append("cluster %d: support row names differ" % gi)
            continue
        for name in sorted(w):
            a, b = np.asarray(w[name]), np.asarray(g[name])
            (parity.cmp_f64 if a.dtype == np.float64 else parity.cmp_int)(name, a, b, "cluster %d support" % gi, bad)
    assert not bad, "%d mismatches, first: %s" % (len(bad), bad[:5])
    assert len(res.batches) >= 3
    stats = {"clusters": len(multi), "spanning": spanning, "batches": len(res.batches)}
    res.free()
    whole.free()
    ctx1.close()
    ctx2.close()
    return stats


def test_device_batches_rule(monkeypatch):
    """the cut of clusters.device_batches equals bench.py's under tightened bounds, and cluster_pass's planner refuses a cluster
    larger than one batch"""
    batch, _ = parity.make_batch(H.SYNTH_PAIRED, 20000, samples=2)
    for span, hits in ((200_000, 10 ** 9), (10 ** 12, 3000), (400_000, 5000)):
        for mod in (bench, CL):
            monkeypatch.setattr(mod, "MAX_BATCH_SPAN", span)
            monkeypatch.setattr(mod, "MAX_BATCH_HITS", hits)
        want = [p.n_bundles for p in bench.device_batches(batch)]
        assert len(want) > 2
        assert [p.n_bundles for p in CL.device_batches(batch)] == want
    with pytest.raises(ValueError, match="cluster 1 alone"):
        CL._cuts([5, 10 ** 13, 5], [1, 1, 1], unit="cluster")


# ---- CPU tier: kernel-logic build ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("free_sources,other_contexts", [(False, False), (True, False), (False, True)])
def test_gather_equals_host_select(emu_lib, free_sources, other_contexts):
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 20000, samples=4)
    check_gather(emu_lib, batch, lt, free_sources, other_contexts)


def test_gather_long_reads(emu_lib):
    batch, lt = parity.make_batch(H.SYNTH_LONG, 2000, samples=2)
    check_gather(emu_lib, batch, lt)


def test_gather_edges_and_errors(emu_lib):
    check_edges(emu_lib)


@pytest.mark.parametrize("mode,templates,samples", [(H.SYNTH_PAIRED, 60000, 4), (H.SYNTH_PAIRED, 40000, 6), (H.SYNTH_SINGLE, 30000, 4)])
def test_cluster_pass_equals_single_batch(emu_lib, mode, templates, samples, monkeypatch):
    print(check_cluster_pass(emu_lib, mode, templates, samples, monkeypatch))


# ---- GPU tier: the CUDA path -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("free_sources,other_contexts", [(False, False), (True, False), (False, True)])
def test_gather_equals_host_select_gpu(free_sources, other_contexts):
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 20000, samples=4)
    check_gather(None, batch, lt, free_sources, other_contexts)


@pytest.mark.gpu
def test_gather_long_reads_gpu():
    batch, lt = parity.make_batch(H.SYNTH_LONG, 3000, samples=2)
    check_gather(None, batch, lt)


@pytest.mark.gpu
def test_gather_many_tiles_gpu():
    """selection and output hits over many look-back tiles"""
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 300000, samples=4, chrom_len=40_000_000)
    st = check_gather(None, batch, lt)
    assert st["bundles"] > 2048 and st["hits"] > 10 ** 6, st


@pytest.mark.gpu
def test_gather_edges_and_errors_gpu():
    check_edges(None)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,templates,samples", [(H.SYNTH_PAIRED, 60000, 4), (H.SYNTH_PAIRED, 40000, 6), (H.SYNTH_SINGLE, 30000, 4)])
def test_cluster_pass_equals_single_batch_gpu(mode, templates, samples, monkeypatch):
    print(check_cluster_pass(None, mode, templates, samples, monkeypatch))
