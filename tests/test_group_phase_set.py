"""Combined phase sets of bundle clusters (agpu_batch_group_phase_set / agpu_group_phase_fetch, gpu.Batch.group_phase_set): the px
of assembler::assemble(vector<bundle*>), the union of the members' phase sets with equal lists counted together, in phase_set::pmap
order.  The model is NumPy over the members' own phase sets (Batch.phase_set), which the parity tests pin to the CPU checkers.
Also: the device ordering of both views through its global-memory path (AGPU_PHASE_SORT_SMEM), the edges and errors of the
call, the cluster pass with phases=True (one process, several output batches; two gloo ranks) and the CLI's cluster_phases.
CPU tier: kernel-logic build; -m gpu: the CUDA path."""
import ctypes as C
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import bench
import fuzz
import parity
from aletsch_b200 import clusters as CL
from aletsch_b200 import gpu as G
from aletsch_b200 import hostlib as H
from aletsch_b200 import run

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def lists_of(d):
    o = d["phase_off"]
    return [tuple(d["phase_val"][o[i]:o[i + 1]].tolist()) for i in range(len(o) - 1)]


def model(ps, members):
    """px.combine(ps) for every member: equal lists summed, ordered like std::map<vector<int32_t>, int> (Python tuples compare
    the same way: element by element, a proper prefix first)"""
    m = {}
    for b in members:
        for l, c in zip(lists_of(ps[b]), ps[b]["phase_cnt"].tolist()):
            m[l] = m.get(l, 0) + c
    items = sorted(m.items())
    off = np.concatenate([[0], np.cumsum([len(l) for l, _ in items])]).astype(np.int32)
    val = np.array([x for l, _ in items for x in l], np.int32)
    return {"phase_off": off, "phase_val": val, "phase_cnt": np.array([c for _, c in items], np.int32)}


def same(a, b):
    return all(np.array_equal(np.asarray(a[k], np.int64), np.asarray(b[k], np.int64)) and len(a[k]) == len(b[k])
               for k in ("phase_off", "phase_val", "phase_cnt"))


def stage5_clusters(ctx, bt, batch, gp):
    """bundle_group::resolve over the region groups of a bridged single batch: its clusters of >= 2 bundles in gv order (as
    test_cluster_pass.single_batch_run forms them)"""
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
    return multi


def single_batch_phases(ctx, batch, gp):
    """the whole job as one device batch: bridge_all, stage 5, group_bridge, graph, phase_set, group_phase_set"""
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.bridge_all(gp)
    multi = stage5_clusters(ctx, bt, batch, gp)
    bt.group_bridge(multi, gp)
    bt.graph(gp)
    ps = bt.phase_set()
    return bt, multi, ps, bt.group_phase_set(multi)


def check_spec(lib, mode, templates, samples):
    ctx = G.Context(0, lib_path=lib)
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    bt, multi, ps, px = single_batch_phases(ctx, batch, gp)
    assert len(multi) >= 5, len(multi)
    assert len(px) == len(multi)
    bad = [gi for gi, (c, d) in enumerate(zip(multi, px)) if not same(model(ps, c), d)]
    assert not bad, "clusters %s differ from the model" % bad[:5]
    # what the data exercised: lists merged from several members, and a proper prefix of another list in one cluster
    merged = prefix = 0
    for c, d in zip(multi, px):
        seen = {}
        for b in c:
            for l in lists_of(ps[b]):
                seen[l] = seen.get(l, 0) + 1
        merged += sum(1 for v in seen.values() if v >= 2)
        ls = lists_of(d)
        prefix += sum(1 for a, b in zip(ls[:-1], ls[1:]) if len(a) < len(b) and b[:len(a)] == a)
    assert merged > 0, "no list is shared by two members"
    assert prefix > 0, "no list is a proper prefix of another in its cluster"
    bt.free()
    ctx.close()
    return {"clusters": len(multi), "merged": merged, "prefix": prefix}


def check_edges(lib):
    ctx = G.Context(0, lib_path=lib)
    # empty bundles every third bundle (unstranded: the reference keeps empty bundles of unstranded libraries only)
    batch = fuzz.random_batch(17, n_bundles=12, max_hits=120, empty_every=3)
    gp = G.default_params(library_type=H.UNSTRANDED)
    bt = ctx.upload(batch.view(), keepalive=batch)
    bt.bridge_all(gp)
    bt.graph(gp)
    # no member phase set yet
    with pytest.raises(G.AgpuError) as ex:
        bt.group_phase_set([[0, 1]])
    assert ex.value.rc == G.AGPU_ERR_ARG
    ps = bt.phase_set()
    nb = batch.n_bundles
    empty = [k for k in range(nb) if len(ps[k]["phase_cnt"]) == 0]
    assert empty, "no bundle without phases"
    # one-member clusters: px = ps
    px = bt.group_phase_set([[k] for k in range(nb)])
    assert all(same(ps[k], px[k]) for k in range(nb))
    # clusters with empty members, and a cluster of only empty ones
    groups = [list(range(0, 5)), list(range(5, 11)), [11]]
    px = bt.group_phase_set(groups)
    assert all(same(model(ps, g), d) for g, d in zip(groups, px))
    assert len(bt.group_phase_set([empty])[0]["phase_cnt"]) == 0
    # no clusters: an empty view
    assert bt.group_phase_set([]) == []

    def fetch_rc():
        v = G.PhaseView()
        return ctx.L.agpu_group_phase_fetch(ctx.h, bt.h, C.byref(v))
    # errors: a bundle out of range, in two clusters, twice in one; nothing is kept afterwards
    for bad in ([[0, nb]], [[-1]], [[0, 1], [1, 2]], [[3, 3]]):
        bt.group_phase_set([[0, 1]])
        assert fetch_rc() == 0
        with pytest.raises(G.AgpuError) as ex:
            bt.group_phase_set(bad)
        assert ex.value.rc == G.AGPU_ERR_ARG
        assert fetch_rc() == G.AGPU_ERR_ARG
    # invalidation: a later phase_set, group_bridge or reset drops the combined phase sets
    strands = fuzz.strand_clusters(batch, np.random.default_rng(3))
    for drop in (lambda: bt._run("phase_set"), lambda: bt.group_bridge(strands, gp), lambda: bt.reset()):
        bt.phase_set()
        bt.group_phase_set([[0, 1]])
        assert fetch_rc() == 0
        drop()
        assert fetch_rc() == G.AGPU_ERR_ARG
    bt.free()
    ctx.close()


def phase_views(lib, mode, templates, samples):
    """member views and combined views of a single-batch run, and the launches of the member fetch"""
    ctx = G.Context(0, lib_path=lib)
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    bt, multi, ps, px = single_batch_phases(ctx, batch, gp)
    l0 = ctx.launches
    G.Batch._phase_view(bt, "agpu_phase_fetch", bt.nb)
    launches = ctx.launches - l0
    bt.free()
    ctx.close()
    return ps, px, launches


def _flat(views):
    return {"%d_%s" % (i, k): np.asarray(d[k]) for i, d in enumerate(views) for k in ("phase_off", "phase_val", "phase_cnt")}


def check_forced_large_path(lib, tmp_path, bound=3, mode=H.SYNTH_PAIRED, templates=20000, samples=3):
    ps, px, launches = phase_views(lib, mode, templates, samples)
    assert max(len(d["phase_cnt"]) for d in ps) > bound and max(len(d["phase_cnt"]) for d in px) > bound
    out = str(tmp_path / "forced.npz")
    body = ("import sys, numpy as np; sys.path.insert(0, 'tests'); import test_group_phase_set as T\n"
            "ps, px, launches = T.phase_views(%r, %r, %d, %d)\n"
            "np.savez(%r, launches=launches, **{'m' + k: v for k, v in T._flat(ps).items()}, **{'x' + k: v for k, v in T._flat(px).items()})\n"
            % (lib, mode, templates, samples, out))
    r = subprocess.run([sys.executable, "-c", body], cwd=ROOT, env=dict(os.environ, AGPU_PHASE_SORT_SMEM=str(bound)), capture_output=True,
                       text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    got = np.load(out)
    want = {"m" + k: v for k, v in _flat(ps).items()}
    want.update({"x" + k: v for k, v in _flat(px).items()})
    assert sorted(want) == sorted(k for k in got.files if k != "launches")
    bad = [k for k in want if want[k].dtype != got[k].dtype or not np.array_equal(want[k], got[k])]
    assert not bad, bad[:5]
    assert int(got["launches"]) > launches, "the global-memory network did not run"


def check_cluster_pass(lib, mode, templates, samples, support, monkeypatch):
    ctx1, ctx2 = G.Context(0, lib_path=lib), G.Context(0, lib_path=lib)
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp = G.default_params(library_type=lt)
    whole, multi, _, px_want = single_batch_phases(ctx1, batch, gp)
    parts = batch.split(3)
    srcs = [ctx2.upload(p.view(), keepalive=p) for p in parts]
    monkeypatch.setattr(CL, "MAX_BATCH_HITS", batch.n_hits // 3 + 1)
    times = {}
    res = CL.cluster_pass(ctx2, parts, srcs, gp, support=support, times=times, phases=True)
    for s in srcs:
        s.free()
    assert len(res.batches) >= 3 and len(res.phases) == len(res.batches) and len(times["phase_set"]) == len(res.batches)
    got_multi = [[int(o[m, 2]) for m in c] for o, cl in zip(res.origin, res.clusters) for c in cl]
    assert got_multi == multi
    spanning = sum(len(set(o[c, 0].tolist())) > 1 for o, cl in zip(res.origin, res.clusters) for c in cl)
    assert spanning > 0, "no cluster spans the parts"
    px_got = [d for p in res.phases for d in p]
    assert len(px_got) == len(px_want)
    bad = [gi for gi in range(len(multi)) if not same(px_want[gi], px_got[gi])]
    assert not bad, "clusters %s differ from the single-batch run" % bad[:5]
    res.free()
    whole.free()
    ctx1.close()
    ctx2.close()


# ---- two gloo ranks ----------------------------------------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, emu, kw, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    import shard_phase_worker
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        q.put((rank, shard_phase_worker.run(lib_path=emu, **kw), None))
    except Exception as e:      # noqa: BLE001
        import traceback
        q.put((rank, None, repr(e) + traceback.format_exc()[-2000:]))
    dist.destroy_process_group()


def run_gloo(emu, world, **kw):
    import torch.multiprocessing as mp
    port = _free_port()
    ctxm = mp.get_context("spawn")
    q = ctxm.Queue()
    procs = [ctxm.Process(target=_gloo_worker, args=(r, world, port, emu, kw, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=900) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, _, err in res:
        assert err is None, "rank %d: %s" % (rank, err)
    return [r for rank, r, _ in sorted(res, key=lambda x: x[0])]


# ---- CLI ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, seed=20261021)
    s = H.Synth(cfg)
    paths = []
    for k in range(3):
        paths.append(str(tmp_path_factory.mktemp("bams") / ("s%d.bam" % k)))
        H.write_bam(paths[-1], s.sample(k, 8000, threads=4), np.array([cfg.chrom_len], np.int32))
    return paths


def check_cli(lib, bams, monkeypatch, capsys):
    if lib:
        monkeypatch.setenv("ALETSCH_GPU_LIB", lib)
    monkeypatch.delenv("WORLD_SIZE", raising=False)

    def cli():
        assert run.main(["--clusters"] + bams) == 0
        return json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    one = cli()
    monkeypatch.setattr(CL, "MAX_BATCH_HITS", one["hits"] // 4)
    cut = cli()
    assert one["device_batches"] == 1 and cut["device_batches"] >= 3
    assert one["cluster_phases"] > 0 and one["cluster_phases"] == cut["cluster_phases"]
    # the same count from the library calls on the job as run.py packs it
    recs, chrom_len = zip(*[H.read_bam(p) for p in bams])
    batch = H.pack(list(recs), H.default_packer_params(H.FR_FIRST), sample_ids=list(range(len(bams))), chrom_len=chrom_len[0],
                   region_length=run.REGION)
    ctx = G.Context(0, lib_path=lib)
    bt, multi, _, px = single_batch_phases(ctx, batch, G.default_params(library_type=H.FR_FIRST))
    assert len(multi) == one["clusters_of_bundles"]
    assert sum(len(d["phase_cnt"]) for d in px) == one["cluster_phases"]
    bt.free()
    ctx.close()


# ---- CPU tier: kernel-logic build --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode,templates,samples", [(H.SYNTH_PAIRED, 40000, 4), (H.SYNTH_SINGLE, 30000, 4), (H.SYNTH_LONG, 3000, 3)])
def test_combined_phase_sets_equal_the_model(emu_lib, mode, templates, samples):
    print(check_spec(emu_lib, mode, templates, samples))


def test_forced_global_memory_ordering(emu_lib, tmp_path):
    check_forced_large_path(emu_lib, tmp_path)


def test_edges_and_errors(emu_lib):
    check_edges(emu_lib)


@pytest.mark.parametrize("support", [False, True])
def test_cluster_pass_phases_equal_single_batch(emu_lib, support, monkeypatch):
    check_cluster_pass(emu_lib, H.SYNTH_PAIRED, 40000 if not support else 20000, 4, support, monkeypatch)


def test_two_ranks_phases_gloo(emu_lib):
    res = run_gloo(emu_lib, 2, samples=5, templates=12000, max_batch_hits=20000)
    assert res[0]["spanning"] > 0 and res[0]["clusters"] > 0


def test_cli_cluster_phases(emu_lib, bams, monkeypatch, capsys):
    check_cli(emu_lib, bams, monkeypatch, capsys)


# ---- GPU tier: the CUDA path -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode,templates,samples", [(H.SYNTH_PAIRED, 60000, 4), (H.SYNTH_SINGLE, 30000, 4), (H.SYNTH_LONG, 3000, 3)])
def test_combined_phase_sets_equal_the_model_gpu(mode, templates, samples):
    print(check_spec(None, mode, templates, samples))


@pytest.mark.gpu
@pytest.mark.parametrize("bound", [3, 16])
def test_forced_global_memory_ordering_gpu(tmp_path, bound):
    check_forced_large_path(None, tmp_path, bound=bound, templates=60000, samples=4)


@pytest.mark.gpu
def test_edges_and_errors_gpu():
    check_edges(None)


@pytest.mark.gpu
@pytest.mark.parametrize("support", [False, True])
def test_cluster_pass_phases_equal_single_batch_gpu(support, monkeypatch):
    check_cluster_pass(None, H.SYNTH_PAIRED, 60000, 4, support, monkeypatch)


@pytest.mark.gpu
def test_cli_cluster_phases_gpu(bams, monkeypatch, capsys):
    check_cli(None, bams, monkeypatch, capsys)
