"""Every agpu_params field away from its default, against every CPU checker present: the per-bundle path (compare_full,
compare_phase_set, compare_revise), the cluster stages (group bridge, group support), stage 5 (agpu_group_resolve_batch on
constructed splice lists against orc_group_resolve_lists) and agpu_similarity_batch against NumPy.  Each case also asserts,
from the fetched views, that it reached the path it is about: a case that silently ran the default path would prove nothing.
Also the regression of min_subregion_gap = 0 (two partial exons [p, p + 1), which the reference asserts against).
CPU tier: kernel-logic build; -m gpu: the CUDA path at larger sizes."""
import ctypes as C

import numpy as np
import pytest

import fuzz
import orclib
import parity
from aletsch_b200 import gpu as G
from aletsch_b200 import hostlib as H

DPW_CMAX = 128          # candidates per vertex the bridging DP keeps in shared memory (k_bridge.h)
SORT_STABLE_MAX = 16    # std::sort is an insertion sort up to 16 elements: ties beyond that take the libstdc++ replay

# (id, changed fields); every case must change the device's outputs on the data (field_case)
KD_CASES = [((1, 1)), ((1, 8)), ((16, 1)), ((16, 8)), ((2, 5))]
FIELD_CASES = [
    ("partition_gap_0", dict(max_reads_partition_gap=0)),
    ("partition_gap_1000", dict(max_reads_partition_gap=1000)),
    ("subregion_gap_1", dict(min_subregion_gap=1)),
    ("subregion_gap_200", dict(min_subregion_gap=200)),
    ("subregion_length_0", dict(min_subregion_length=0)),
    ("subregion_length_200", dict(min_subregion_length=200)),
    ("subregion_overlap_0", dict(min_subregion_overlap=0.0)),
    ("subregion_overlap_10", dict(min_subregion_overlap=10.0)),
    ("edge_weight_0", dict(min_guaranteed_edge_weight=0.0)),
    ("edge_weight_1", dict(min_guaranteed_edge_weight=1.0)),
    ("corner_small", dict(bridge_dp_solution_size=1, bridge_dp_stack_size=1, max_reads_partition_gap=0, min_subregion_gap=1,
                          min_subregion_length=0, bridge_end_relaxing=0)),
    ("corner_large", dict(bridge_dp_solution_size=16, bridge_dp_stack_size=8, max_reads_partition_gap=1000, min_subregion_gap=200,
                          min_guaranteed_edge_weight=1.0, insertsize_low=0, insertsize_high=1000000, bridge_end_relaxing=1000)),
]
INSERT_CASES = [dict(insertsize_low=0, insertsize_high=1000000), dict(insertsize_low=300, insertsize_high=310),
                dict(insertsize_low=80, insertsize_high=500), dict(bridge_end_relaxing=0), dict(bridge_end_relaxing=1000)]


# ---------------------------------------------------------------------------------------------------------------- data

def per_bundle_data(large):
    """(name, batch, library type): a synthetic paired batch, a long-read batch and fuzz batches (one pair-heavy, one with
    coarse exon grid: in-degrees up to a few dozen)"""
    out = []
    b, lt = parity.make_batch(H.SYNTH_PAIRED, 30000 if large else 6000)
    out.append(("paired", b, lt))
    b, lt = parity.make_batch(H.SYNTH_LONG, 3000 if large else 600)
    out.append(("long", b, lt))
    for seed in ((0, 1, 2, 5) if large else (0, 1)):
        fb = fuzz.random_batch(seed, n_bundles=8 if large else 5, max_hits=250, exon_grid=(seed % 2 == 0), pair_heavy=(seed % 2 == 1))
        out.append(("fuzz%d" % seed, fb, H.FR_FIRST))
    # complete-DAG bundles: the bridging DP meets vertices with hundreds of candidates (see dp_rows)
    dags = [fuzz.dag_bundle(20), fuzz.dag_bundle(12, strand="-", reads_per_junction=2)]
    if large:
        dags.append(fuzz.dag_bundle(26, reads_per_junction=3))
    out.append(("dag", fuzz.pack_bundles(dags), H.FR_FIRST))
    return out


def device_outputs(ctx, batch, gp):
    """what the device computes on the per-bundle path, flattened: graph, clusters / bridged counts, phase sets, revision"""
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.bridge_all(gp)
    counts = bt.counts()
    fr = bt.fetch_fragments()
    bt.graph(gp)
    gr = bt.fetch_graph()
    ph = bt.phase_set()
    rv = bt.revise(gp)
    bt.free()
    out = {"clusters": counts["clusters"], "bridged": counts["bridged"]}
    for k in range(batch.n_bundles):
        for d in (gr[k], ph[k], rv[k]):
            for n, a in d.items():
                out["%d %s" % (k, n)] = np.asarray(a)
        out["%d frgs" % k] = fr[k]["frgs"]
    return out, gr


def differs(a, b):
    return a.keys() != b.keys() or any(not np.array_equal(a[n], b[n]) for n in a)


def locate_vertex(vl, vr, p):
    """locate_vertex (k_cluster.h): the inner vertex holding position p, or -1"""
    a, b, m = 1, len(vl) - 1, -1
    while a < b:
        mid = (a + b) // 2
        if vl[mid] <= p < vr[mid]:
            m = mid
            break
        if p < vl[mid]:
            b = mid
        else:
            a = mid + 1
    if m < 0:
        m = b
    return m if vl[m] <= p < vr[m] else -1


def dp_rows(gr, cl, K, D, relax):
    """the candidate lists of the bridging DP, replayed on the host from one bundle's fetched graph and cluster views:
    bridging vertices with end relaxing (build_bridging_vertices), piers and pier groups (build_piers), then per group, strand
    pass and vertex the candidates update_stack makes from every in-edge's kept entries (dynamic_programming).  Yields
    (number of candidates, whether two of them compare equal under entry_compare) per DP row.  Only (stack, length) values
    matter here: entries that compare equal have the same values, so which of them the sort keeps changes no count."""
    vert = gr["vert"].reshape(-1, 5)
    vl, vr = vert[:, 0].tolist(), vert[:, 1].tolist()
    nv = len(vl)
    n = nv - 1
    real = set()
    ins = [[] for _ in range(nv)]
    for (s, t, st), w in zip(gr["edge"].reshape(-1, 3).tolist(), gr["edge_d"].tolist()):
        real.add((s, t))
        ins[t].append((s, st, int(w)))

    def pseudo(i):
        return 1 <= i < nv - 2 and (i, i + 1) not in real

    def continuous(x):
        return ((x, x + 1) in real or pseudo(x)) and vr[x] == vl[x + 1]

    bo = cl["clu_bounds"].reshape(-1, 4)
    groups = {}
    for c in range(len(bo)):
        bd1, bd2 = int(bo[c, 1]), int(bo[c, 2])
        c1 = cl["clu_c1_val"][cl["clu_c1_off"][c]:cl["clu_c1_off"][c + 1]]
        c2 = cl["clu_c2_val"][cl["clu_c2_off"][c]:cl["clu_c2_off"][c + 1]]
        v1, v2 = locate_vertex(vl, vr, bd1 - 1), locate_vertex(vl, vr, bd2)
        if 1 < v1 < n and continuous(v1 - 1) and bd1 - vl[v1] <= relax and not (len(c1) and c1[-1] >= vl[v1]):
            v1 -= 1
        if 0 < v2 < n - 1 and continuous(v2) and vr[v2] - bd2 <= relax and not (len(c2) and c2[0] <= vr[v2]):
            v2 += 1
        if 0 <= v1 < v2:
            groups[v1] = max(groups.get(v1, v2), v2)
    passes = {ord("."): (1, 2), ord("+"): (1,), ord("-"): (2,)}.get(int(gr["graph"][0]), ())
    for k1, k2 in sorted(groups.items()):
        for strand in passes:
            rows = {k1: [((999999,) * D, vr[k1] - vl[k1])]}
            for k in range(k1 + 1, k2 + 1):
                edges = [(j, w) for j, st, w in ins[k] if (st == 0 or st == strand) and j >= k1]
                if pseudo(k - 1):
                    edges.append((k - 1, 0))
                cand = []
                for j, w in edges:
                    for stack, ln in rows[j]:
                        out, a, q = [0] * D, 0, 0
                        while a < D and q < D:
                            if a == q and stack[a] > w:
                                out[q] = w
                                q += 1
                                if q >= D:
                                    break
                            out[q] = stack[a]
                            a += 1
                            q += 1
                        cand.append((tuple(out), ln + vr[k] - vl[k]))
                keys = [(tuple(-x for x in st), ln) for st, ln in cand]
                yield len(cand), len(set(keys)) < len(keys)
                rows[k] = [cand[i] for i in sorted(range(len(cand)), key=keys.__getitem__)[:K]]


def dp_paths(ctx, batch, lt, K, D):
    """(rows with more than DPW_CMAX candidates, rows with 17..DPW_CMAX candidates and a tie) of the bridging DP on a batch"""
    gp = G.default_params(library_type=lt, bridge_dp_solution_size=K, bridge_dp_stack_size=D)
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.evidence(gp)
    ev = bt.fetch_evidence(batch.a["bundle_hit_off"])
    bt.fragments()
    bt.graph(gp)
    gr = bt.fetch_graph()
    bt.cluster(gp)
    cl = bt.fetch_clusters(ev)
    bt.free()
    big = tie = 0
    for k in range(batch.n_bundles):
        for nc, t in dp_rows(gr[k], cl[k], K, D, gp.bridge_end_relaxing):
            big += nc > DPW_CMAX
            tie += SORT_STABLE_MAX < nc <= DPW_CMAX and t
    return big, tie


def check_parity(ctx, checkers, batch, gp, op, where):
    assert checkers, "no CPU checker"
    for name, chk in checkers.items():
        for f in (parity.compare_full, parity.compare_phase_set, parity.compare_revise):
            bad = f(ctx, batch, chk, gp, op)
            assert not bad, "%s %s vs %s: %d mismatches: %s" % (where, f.__name__, name, len(bad), bad[:3])


class Sweep:
    """the data of one tier and the default run on it (computed once)"""

    def __init__(self, ctx, large):
        self.ctx = ctx
        self.data = per_bundle_data(large)
        self.base = {}
        for name, b, lt in self.data:
            self.base[name] = device_outputs(ctx, b, G.default_params(library_type=lt))[0]

    def run_case(self, checkers, kw):
        """parity on every batch; returns per batch (outputs, graph views, whether they differ from the default run)"""
        res = {}
        for name, b, lt in self.data:
            gp, op = parity.params_pair(lt, **kw)
            check_parity(self.ctx, checkers, b, gp, op, "%s %s" % (name, kw))
            out, gr = device_outputs(self.ctx, b, gp)
            res[name] = (out, gr, differs(out, self.base[name]))
        return res


def kd_case(sweep, checkers, K, D):
    """parity at K, D; the candidate counts of the DP, replayed from the fetched views, show that the std::sort tie replay ran
    (more than 16 candidates with a tie) and, at K = 16, the global-memory candidates (more than DPW_CMAX).  At K <= 2 the
    latter needs more in-edges inside one bridging range than the shared in-edge slice holds, so it is not asserted there."""
    res = sweep.run_case(checkers, dict(bridge_dp_solution_size=K, bridge_dp_stack_size=D))
    assert any(r[2] for r in res.values()), "K, D = %d, %d changed nothing" % (K, D)
    big = tie = 0
    for name, b, lt in sweep.data:
        x, y = dp_paths(sweep.ctx, b, lt, K, D)
        big += x
        tie += y
    assert tie > 0, "no DP row with more than 16 candidates and a tie at K, D = %d, %d" % (K, D)
    if K >= 16:
        assert big > 0, "no DP row with more than %d candidates at K, D = %d, %d" % (DPW_CMAX, K, D)


def field_case(sweep, checkers, kw):
    res = sweep.run_case(checkers, kw)
    assert any(r[2] for r in res.values()), "%s changed nothing on the data" % kw


def junction_thresholds(sweep, checkers):
    """normal_junction_threshold / extend_junction_threshold: neither the device path nor the restatement reads them, so the
    outputs must equal the default run's.  That is all the restatement can establish.  SURVEY.md lists both fields among the
    reference's reads, so whether ignoring them is right on this path is settled only where the reference build (checker
    'ref', oracle/_ref) is present: there the same cases compare the device with the reference's own code."""
    for v in (1, 1000):
        res = sweep.run_case(checkers, dict(normal_junction_threshold=v, extend_junction_threshold=v))
        assert not any(r[2] for r in res.values())


def insert_cases(sweep, checkers):
    bridged = []
    for kw in INSERT_CASES:
        res = sweep.run_case(checkers, kw)
        bridged.append(tuple(int(r[0]["bridged"]) for r in res.values()))
    assert len(set(bridged)) >= 4, "the insert-size bounds and bridge_end_relaxing hardly change the bridged counts: %s" % bridged


def bad_kd(ctx, batch, lt):
    """out-of-range K or D: agpu_batch_bridge refuses (AGPU_ERR_ARG); the batch can still be reset and bridged at the defaults"""
    gp0 = G.default_params(library_type=lt)
    want, _ = device_outputs(ctx, batch, gp0)
    for K, D in ((0, 5), (17, 5), (10, 0), (10, 9)):
        bt = ctx.upload(batch.view(), keepalive=batch)
        bt.evidence(gp0)
        bt.fragments()
        bt.graph(gp0)
        bt.cluster(gp0)
        with pytest.raises(G.AgpuError) as e:
            bt.bridge(G.default_params(library_type=lt, bridge_dp_solution_size=K, bridge_dp_stack_size=D))
        assert e.value.rc == G.AGPU_ERR_ARG
        bt.reset()
        bt.bridge_all(gp0)
        assert bt.counts()["bridged"] == want["bridged"]
        bt.free()


# ---------------------------------------------------------------------------------------------------------------- gap 0

def gap0_regression(ctx, checkers):
    """fuzz seed 3 at min_subregion_gap = 0: bundles 0, 4, 5 and 7 each get a 1-bp region between a junction end and a junction
    start with no coverage, and so both stubs of build_partial_exons, [p, p + 1) twice.  link_partial_exons asserts that no two
    partial exons share a bound (rnacore/graph_builder.cc:255-258): the device reports it, as it reports a junction without a
    partial exon, and every stage of the restatement that builds the graph fails on exactly those bundles.  At gap 1 the
    region is smoothed over."""
    fb = fuzz.random_batch(3, n_bundles=8, max_hits=250, exon_grid=False)
    gp, op = parity.params_pair(H.FR_FIRST, min_subregion_gap=0)
    bt = ctx.upload(fb.view(), keepalive=fb)
    bt.evidence(gp)
    with pytest.raises(G.AgpuError) as e:
        bt.graph(gp)
    assert "4 violation(s) of: two partial exons with a common bound" in str(e.value)
    bt.free()
    if "orc" in checkers:
        chk = checkers["orc"]
        for stage in ("graph", "bridge", "phase", "revise"):
            rcs = []
            for k in range(fb.n_bundles):
                h = chk.new_bundle(fb.bundle(k), op)
                chk.run(h, "evidence")
                chk.run(h, "fragments")
                rcs.append(chk.run(h, stage)[0])
                chk.free_bundle(h)
            assert [k for k, rc in enumerate(rcs) if rc < 0] == [0, 4, 5, 7], (stage, rcs)
    # gap 1 fills the 1-bp stretch: one partial exon there, and everything matches
    gp1, op1 = parity.params_pair(H.FR_FIRST, min_subregion_gap=1)
    for name, chk in checkers.items():
        bad = parity.compare_full(ctx, fb, chk, gp1, op1)
        assert not bad, "%s: %s" % (name, bad[:3])


def gap0_sweep(ctx, checkers, large):
    """min_subregion_gap = 0 on batches where no such 1-bp region arises: full parity, and the outputs differ from the default
    run on the fuzz batches (the synthetic coverage has no short gaps between splice sites)"""
    data = per_bundle_data(large)[:2]
    for seed in ((0, 1, 2, 5) if large else (0, 1, 2)):
        data.append(("fuzz%d" % seed, fuzz.random_batch(seed, n_bundles=8, max_hits=250 if seed % 2 else 70, exon_grid=(seed % 2 == 0)),
                     H.FR_FIRST))
    changed = False
    for name, b, lt in data:
        gp, op = parity.params_pair(lt, min_subregion_gap=0)
        check_parity(ctx, checkers, b, gp, op, name + " gap 0")
        changed |= differs(device_outputs(ctx, b, gp)[0], device_outputs(ctx, b, G.default_params(library_type=lt))[0])
    assert changed


def fr_second_batch(templates):
    """the synthetic paired reads as an fr-secondstrand library tags them (XS '+' and '-' swapped), packed for FR_SECOND"""
    cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, seed=20260101)
    rec = H.Synth(cfg).sample(0, templates, threads=4)
    x = rec["xs"].copy()
    rec["xs"] = np.where(x == ord("+"), ord("-"), np.where(x == ord("-"), ord("+"), x)).astype(np.uint8)
    return H.pack([rec], H.default_packer_params(H.FR_SECOND))


def fr_second(ctx, checkers, large):
    """library_type FR_SECOND on a batch packed for it: bundles with spliced hits on both strands, then every stage"""
    b = fr_second_batch(20000 if large else 5000)
    assert b.n_bundles > 10, b.n_bundles
    spliced = sum(any((c & 0xF) == fuzz.N for c in b.a["cigar"][b.a["cigar_off"][i]:b.a["cigar_off"][i + 1]]) for i in range(b.n_hits))
    assert spliced > 100, spliced
    starts = b.a["strand"][b.a["bundle_hit_off"][:-1]]
    assert {ord("+"), ord("-")} <= set(starts.tolist())
    gp, op = parity.params_pair(H.FR_SECOND)
    check_parity(ctx, checkers, b, gp, op, "fr_second")


# ---------------------------------------------------------------------------------------------------------------- clusters

def sampled_fuzz(seed, n_bundles):
    """a fuzz batch whose bundles carry random samples 0-2, so clusters hold several bundles of one sample"""
    fb = fuzz.random_batch(seed, n_bundles=n_bundles, max_hits=120, exon_grid=True)
    rng = np.random.default_rng(seed + 100)
    fb.a["bundle_sample"] = rng.integers(0, 3, fb.n_bundles).astype(np.int32)
    groups = fuzz.strand_clusters(fb, rng)
    repeats = sum(len(g) - len(set(fb.a["bundle_sample"][g].tolist())) for g in groups)
    assert repeats > 0, "no cluster holds two bundles of one sample"
    return fb, groups


def cluster_data(large):
    b, lt = parity.make_batch(H.SYNTH_PAIRED, 30000 if large else 12000, samples=4)
    out = [("multi-sample", b, lt, parity.locus_groups(b, max_groups=12 if large else 5))]
    for seed in ((7, 8, 9) if large else (7,)):
        fb, groups = sampled_fuzz(seed, 16 if large else 10)
        out.append(("fuzz%d" % seed, fb, H.FR_FIRST, groups))
    return out


def cluster_kd(ctx, checkers, large, K, D):
    for name, b, lt, groups in cluster_data(large):
        gp, op = parity.params_pair(lt, bridge_dp_solution_size=K, bridge_dp_stack_size=D)
        for cname, chk in checkers.items():
            bad = parity.compare_group_bridge(ctx, b, chk, gp, op, groups)
            assert not bad, "%s group bridge vs %s: %s" % (name, cname, bad[:3])
            bad = parity.compare_group_support(ctx, b, chk, gp, op, groups)
            assert not bad, "%s group support vs %s: %s" % (name, cname, bad[:3])


def member_edges(ctx, b, gp, groups):
    bt = ctx.upload(b.view(), keepalive=b)
    bt.bridge_all(gp)
    bt.group_bridge(groups, gp)
    got = bt.group_support(groups, gp)
    bt.free()
    return [np.asarray(d[n]) for d in got for n in sorted(d) if n.endswith("sup_edge")]


def boundary_distance(ctx, checkers, large):
    """max_group_boundary_distance of group_start_boundaries / group_end_boundaries (k_sup_regroup): parity at 0, 100 and
    10^7, and the members' regrouped graphs differ between 0 and 10^7.  A log ratio of 0.5 lets the revision add enough start
    and end boundaries that several fall in one continuous stretch."""
    changed = False
    for name, b, lt, groups in cluster_data(large):
        for dist in (0, 100, 10 ** 7):
            gp, op = parity.params_pair(lt, max_group_boundary_distance=dist, min_boundary_log_ratio=0.5)
            for cname, chk in checkers.items():
                bad = parity.compare_group_support(ctx, b, chk, gp, op, groups)
                assert not bad, "%s distance %d vs %s: %s" % (name, dist, cname, bad[:3])
        e0 = member_edges(ctx, b, G.default_params(library_type=lt, max_group_boundary_distance=0, min_boundary_log_ratio=0.5), groups)
        e1 = member_edges(ctx, b, G.default_params(library_type=lt, max_group_boundary_distance=10 ** 7, min_boundary_log_ratio=0.5),
                          groups)
        changed |= len(e0) != len(e1) or any(not np.array_equal(x, y) for x, y in zip(e0, e1))
    assert changed, "max_group_boundary_distance 0 and 10^7 regroup the same boundaries"


# ---------------------------------------------------------------------------------------------------------------- stage 5

def resolve_lists(chk, lists, params):
    """orc_group_resolve_lists: the restatement's bundle_group::resolve on given lists; gvv order, indices local"""
    L = chk.lib
    f = L.orc_group_resolve_lists
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(orclib.Params), C.c_void_p]
    off = np.zeros(len(lists) + 1, np.int64)
    for i, l in enumerate(lists):
        off[i + 1] = off[i] + len(l)
    val = np.ascontiguousarray(np.concatenate([np.asarray(l, np.int32) for l in lists] + [np.zeros(1, np.int32)]), np.int32)
    bag = L.orc_bag_new()
    assert f(len(lists), off.ctypes.data, val.ctypes.data, C.byref(params), bag) == 0
    d = chk.bag_to_dict(bag)
    L.orc_bag_free(bag)
    o, v = d["gvv_off"], d["gvv_val"]
    return [v[o[i]:o[i + 1]].tolist() for i in range(len(o) - 1)]


def resolve_checker(checkers):
    if "orc" not in checkers:
        pytest.skip("the restatement (oracle/liboracle.so) is not built")
    return checkers["orc"]


def check_groups(ctx, chk, groups, **kw):
    """agpu_group_resolve_batch on all groups in one call == orc_group_resolve_lists group by group; returns the clusterings"""
    gp = G.default_params(**kw)
    op = orclib.default_params(**kw)
    got = G.group_resolve_batch(ctx, groups, gp)
    for gi, grp in enumerate(groups):
        want = resolve_lists(chk, grp, op) if len(grp) else []
        assert got[gi] == want, "group %d (%d lists) %s: device %s vs checker %s" % (gi, len(grp), kw, got[gi][:6], want[:6])
    return got


def pair(c, n_small, n_big, base=1000):
    """two sorted lists of n_small and n_big splice positions with exactly c in common"""
    a = base + 2 * np.arange(n_small)
    b = np.concatenate([a[:c], base + 100000 + 2 * np.arange(n_big - c)])
    return [np.sort(a).astype(np.int32), np.sort(b).astype(np.int32)]


def threshold_pairs(ctx, checkers):
    """pairs whose ratio c / min(|A|, |B|) is exactly the threshold join; one common splice less does not"""
    chk = resolve_checker(checkers)
    for c, n, s in ((1, 5, 0.2), (3, 10, 0.3), (2, 4, 0.5), (4, 4, 1.0)):
        for m in (c, c - 1):
            for thr_field in ("min_grouping_similarity", "max_grouping_similarity"):
                kw = dict(min_grouping_similarity=s, max_grouping_similarity=max(s, 0.8)) if thr_field == "min_grouping_similarity" \
                    else dict(min_grouping_similarity=1.0, max_grouping_similarity=s)
                got = check_groups(ctx, chk, [pair(m, n, n + 3)], **kw)
                joined = (m == c) and (m > 0)
                assert got[0] == ([[0, 1]] if joined else [[0], [1]]), (c, n, s, m, kw, got)


def junction_cap(ctx, checkers):
    """lists of 2 * max_num_junctions_to_combine splices take part, longer ones do not"""
    chk = resolve_checker(checkers)
    for cap in (1, 3, 5):
        at = (1000 + 2 * np.arange(2 * cap)).astype(np.int32)
        above = np.sort(np.concatenate([at, [900000, 900002]])).astype(np.int32)
        above1 = np.sort(np.concatenate([at, [900000]])).astype(np.int32)
        grp = [at, at.copy(), above, above1]
        got = check_groups(ctx, chk, [grp], max_num_junctions_to_combine=cap)
        assert got[0] == [[0, 1], [2], [3]], (cap, got)


def random_groups(rng, sizes, pool_size=60, max_len=14):
    groups = []
    for g in sizes:
        pool = np.sort(rng.choice(200000, size=pool_size, replace=False)).astype(np.int32)
        groups.append([np.sort(rng.choice(pool, size=int(rng.integers(0, max_len + 1)), replace=False)).astype(np.int32)
                       for _ in range(g)])
    return groups


def similarity_ranges(ctx, checkers, sizes):
    """random groups on both sides of the one-CTA tile (32) and of the one-CTA group limit (192), several per call, over the
    grouping thresholds, the size cap and the junction cap"""
    chk = resolve_checker(checkers)
    rng = np.random.default_rng(23)
    groups = random_groups(rng, sizes)
    seen = set()
    for hi in (0.1, 0.5, 1.0):
        for lo in (0.0, 1.0):
            for kw in (dict(), dict(max_group_size=4), dict(max_num_junctions_to_combine=3)):
                got = check_groups(ctx, chk, groups, max_grouping_similarity=hi, min_grouping_similarity=lo, **kw)
                seen.add(tuple(len(g) for g in got))
    assert len(seen) > 3, "the thresholds do not change the clusterings"


def similarity_batch(ctx, sizes):
    """agpu_similarity_batch: every upper-triangle count == |intersect1d|; groups above 192 lists take agpu_similarity"""
    rng = np.random.default_rng(5)
    groups = random_groups(rng, sizes, pool_size=80, max_len=30)
    got = ctx.similarity_batch(groups)
    assert len(got) == len(groups)
    for grp, c in zip(groups, got):
        assert c.shape == (len(grp), len(grp))
        want = np.zeros_like(c)
        for i in range(len(grp)):
            for j in range(i + 1, len(grp)):
                want[i, j] = len(np.intersect1d(grp[i], grp[j]))
        iu = np.triu_indices(len(grp), 1)
        assert np.array_equal(c[iu], want[iu])
        if len(grp) >= 33:
            assert want[iu].max() > 0


# ---------------------------------------------------------------------------------------------------------------- CPU tier

@pytest.fixture(scope="module")
def ctx(emu_lib):
    c = G.Context(0, lib_path=emu_lib)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sweep(ctx):
    return Sweep(ctx, large=False)


@pytest.mark.parametrize("K,D", KD_CASES)
def test_dp_sizes(sweep, checkers, K, D):
    kd_case(sweep, checkers, K, D)


@pytest.mark.parametrize("kw", [c[1] for c in FIELD_CASES], ids=[c[0] for c in FIELD_CASES])
def test_field(sweep, checkers, kw):
    field_case(sweep, checkers, kw)


def test_junction_thresholds(sweep, checkers):
    junction_thresholds(sweep, checkers)


def test_insert_size_and_end_relaxing(sweep, checkers):
    insert_cases(sweep, checkers)


def test_out_of_range_dp_sizes(ctx):
    b, lt = parity.make_batch(H.SYNTH_PAIRED, 3000)
    bad_kd(ctx, b, lt)


def test_subregion_gap_0_regression(ctx, checkers):
    gap0_regression(ctx, checkers)


def test_subregion_gap_0(ctx, checkers):
    gap0_sweep(ctx, checkers, large=False)


def test_fr_second(ctx, checkers):
    fr_second(ctx, checkers, large=False)


@pytest.mark.parametrize("K,D", [(16, 8), (1, 1)])
def test_cluster_stages_dp_sizes(ctx, checkers, K, D):
    cluster_kd(ctx, checkers, False, K, D)


def test_group_boundary_distance(ctx, checkers):
    boundary_distance(ctx, checkers, False)


def test_similarity_threshold_pairs(ctx, checkers):
    threshold_pairs(ctx, checkers)


def test_junction_cap(ctx, checkers):
    junction_cap(ctx, checkers)


def test_group_sizes_and_thresholds(ctx, checkers):
    similarity_ranges(ctx, checkers, (0, 1, 2, 31, 32, 33, 5))


def test_similarity_batch(ctx):
    similarity_batch(ctx, (0, 1, 2, 33, 192, 193))


# ---------------------------------------------------------------------------------------------------------------- GPU tier

@pytest.fixture(scope="module")
def gctx():
    c = G.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def gsweep(gctx):
    return Sweep(gctx, large=True)


@pytest.mark.gpu
@pytest.mark.parametrize("K,D", KD_CASES)
def test_dp_sizes_gpu(gsweep, checkers, K, D):
    kd_case(gsweep, checkers, K, D)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [c[1] for c in FIELD_CASES], ids=[c[0] for c in FIELD_CASES])
def test_field_gpu(gsweep, checkers, kw):
    field_case(gsweep, checkers, kw)


@pytest.mark.gpu
def test_junction_thresholds_gpu(gsweep, checkers):
    junction_thresholds(gsweep, checkers)


@pytest.mark.gpu
def test_insert_size_and_end_relaxing_gpu(gsweep, checkers):
    insert_cases(gsweep, checkers)


@pytest.mark.gpu
def test_out_of_range_dp_sizes_gpu(gctx):
    b, lt = parity.make_batch(H.SYNTH_PAIRED, 20000)
    bad_kd(gctx, b, lt)


@pytest.mark.gpu
def test_subregion_gap_0_regression_gpu(gctx, checkers):
    gap0_regression(gctx, checkers)


@pytest.mark.gpu
def test_subregion_gap_0_gpu(gctx, checkers):
    gap0_sweep(gctx, checkers, large=True)


@pytest.mark.gpu
def test_fr_second_gpu(gctx, checkers):
    fr_second(gctx, checkers, large=True)


@pytest.mark.gpu
@pytest.mark.parametrize("K,D", [(16, 8), (1, 1)])
def test_cluster_stages_dp_sizes_gpu(gctx, checkers, K, D):
    cluster_kd(gctx, checkers, True, K, D)


@pytest.mark.gpu
def test_group_boundary_distance_gpu(gctx, checkers):
    boundary_distance(gctx, checkers, True)


@pytest.mark.gpu
def test_similarity_threshold_pairs_gpu(gctx, checkers):
    threshold_pairs(gctx, checkers)


@pytest.mark.gpu
def test_junction_cap_gpu(gctx, checkers):
    junction_cap(gctx, checkers)


@pytest.mark.gpu
def test_group_sizes_and_thresholds_gpu(gctx, checkers):
    similarity_ranges(gctx, checkers, (0, 1, 2, 31, 32, 33, 191, 192, 193, 7))


@pytest.mark.gpu
def test_similarity_batch_gpu(gctx):
    similarity_batch(gctx, (0, 1, 2, 33, 192, 193, 400))
