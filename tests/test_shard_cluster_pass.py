"""The cross-sample cluster pass with samples ingested on different ranks (shard.cluster_pass_sharded): the planner, the exchange of
bundles between ranks and the pass on every cluster's owner.  The oracle is the whole job run as one device batch
(test_cluster_pass.single_batch_run).  CPU tier: gloo on the kernel-logic build, ranks spawned like test_shard_gloo.py.  GPU tier: the
pointer view of a batch's device columns on one GPU; NCCL and the CLI under torchrun on two (skipped with fewer)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

import parity
import test_cluster_pass as T
from aletsch_b200 import clusters as CL
from aletsch_b200 import gpu as G
from aletsch_b200 import hostlib as H
from aletsch_b200 import shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
    import shard_cluster_worker
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        q.put((rank, shard_cluster_worker.run("gloo", lib_path=emu, **kw), None))
    except Exception as e:      # noqa: BLE001
        import traceback
        q.put((rank, None, repr(e) + traceback.format_exc()[-2000:]))
    dist.destroy_process_group()


def run_gloo(emu, world, **kw):
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


# ---- planner (no process group) ----------------------------------------------------------------------------------------------

def random_job(seed, n=400, world=3):
    rng = np.random.default_rng(seed)
    sample = rng.integers(0, 7, n)
    keys = (sample.astype(np.int64) << 32) | np.arange(n)
    region = rng.integers(0, 12, n).astype(np.int64) << 8
    cluster = rng.integers(0, 40, n)
    return dict(keys=keys, region=region, cluster=cluster, owner=sample % world, hits=rng.integers(1, 5000, n),
                span=rng.integers(300, 20000, n))


def test_plan_is_the_same_from_every_rank():
    job = random_job(1)
    want = shard.plan_clusters(world=3, **job)
    for seed in range(3):
        perm = np.random.default_rng(seed).permutation(len(job["keys"]))
        got = shard.plan_clusters(world=3, **{k: v[perm] for k, v in job.items()})
        assert np.array_equal(got.dest, want.dest) and np.array_equal(got.load, want.load)
        for r in range(3):
            assert np.array_equal(job["keys"][want.rows[r]], job["keys"][perm][got.rows[r]])
            assert np.array_equal(got.cstart[r], want.cstart[r])


def test_plan_layout_singletons_and_lpt_bound():
    job = random_job(2, world=3)
    p = shard.plan_clusters(world=3, **job)
    seen = np.concatenate(p.rows)
    assert np.array_equal(np.sort(seen), np.arange(len(job["keys"])))
    seed = np.zeros(3, np.int64)
    for r in range(3):
        rows, st = p.rows[r], p.cstart[r]
        # members in (region, key) order, clusters in (region, cluster) order
        order = np.lexsort((job["keys"][rows], job["cluster"][rows], job["region"][rows]))
        assert np.array_equal(order, np.arange(len(rows)))
        for a, b in zip(st[:-1], st[1:]):
            m = rows[a:b]
            assert len(set(job["region"][m])) == 1 and len(set(job["cluster"][m])) == 1
            if b - a == 1:
                assert job["owner"][m[0]] == r, "a singleton moved"
                seed[r] += job["hits"][m[0]]
    assert p.size.sum() == len(job["keys"]) and (p.size == 1).any() and (p.size >= 2).any()
    w = np.array([job["hits"][p.rows[r]].sum() for r in range(3)])
    assert np.array_equal(w, p.load)
    multi_max = max(int(job["hits"][p.rows[r][a:b]].sum()) for r in range(3) for a, b in zip(p.cstart[r][:-1], p.cstart[r][1:]) if b - a >= 2)
    assert p.load.max() <= max(seed.max(), p.load.min() + multi_max)       # LPT bound with seeded loads


def test_assign_units_seeded_load():
    rng = np.random.default_rng(5)
    w = rng.integers(1, 1000, 200)
    for world in (2, 3, 8):
        seed = rng.integers(0, 20000, world)
        r = shard.assign_units(w, world, seed)
        load = seed + np.array([w[r == k].sum() for k in range(world)])
        assert load.max() <= max(seed.max(), load.min() + w.max())
    assert list(shard.assign_units([5, 5, 5], 2, [10, 0])) == [1, 1, 0]
    assert list(shard.assign_units([5, 5, 5], 2)) == list(shard.assign_units([5, 5, 5], 2, [0, 0]))


def test_plan_rejects_an_oversized_cluster(monkeypatch):
    job = random_job(3, world=2)
    monkeypatch.setattr(CL, "MAX_BATCH_HITS", 12000)
    with pytest.raises(ValueError, match="alone exceeds the batching rule"):
        shard.plan_clusters(world=2, **job)


def test_gather_packed_four_argument_call():
    """bench.py's call: one extra column, no process group"""
    off = np.array([0, 2, 5], np.int64)
    val = np.array([1, 2, 3, 4, 5], np.int32)
    keys = np.array([7, 9], np.int64)
    regs = np.array([100, 200], np.int64)
    o, v, k, x, owner, nbytes = shard.gather_packed(off, val, keys, regs)
    assert np.array_equal(o, off) and np.array_equal(v, val) and np.array_equal(k, keys) and np.array_equal(x, regs)
    assert x.shape == (2,) and np.array_equal(owner, [0, 0]) and nbytes == 0
    cols = np.stack([regs, regs + 1], axis=1)
    assert np.array_equal(shard.gather_packed(off, val, keys, cols)[3], cols)


# ---- CPU tier: kernel-logic build --------------------------------------------------------------------------------------------

def test_no_process_group_equals_cluster_pass(emu_lib):
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 20000, samples=4)
    gp = G.default_params(library_type=lt)
    ctx = G.Context(0, lib_path=emu_lib)
    parts = batch.split(3)
    keys = (batch.a["bundle_sample"].astype(np.int64) << 32) | np.arange(batch.n_bundles)
    want = CL.cluster_pass(ctx, parts, [ctx.upload(p.view(), keepalive=p) for p in parts], gp, support=True)
    times = {}
    got = shard.cluster_pass_sharded(ctx, parts, [ctx.upload(p.view(), keepalive=p) for p in parts], keys, gp, support=True, times=times)
    assert {"evidence", "signatures", "stage5", "plan", "exchange", "gather", "bridge_all", "group_bridge", "group_support"} <= set(times)
    assert got.n_clusters == want.n_clusters and got.clusters == want.clusters and len(got.batches) == len(want.batches)
    assert got.exchange["bytes_sent"] == 0 and got.exchange["bytes_received"] == 0
    nh = np.diff(batch.a["bundle_hit_off"])
    for gb, wb, go, wo, gs, ws in zip(got.batches, want.batches, got.origin, want.origin, got.support, want.support):
        assert np.array_equal(go[:, 0], np.zeros(len(go))) and np.array_equal(go[:, 1], keys[wo[:, 2]])
        assert np.array_equal(go[:, 2:], wo[:, :2])
        loc = np.concatenate([[0], np.cumsum(nh[wo[:, 2]])])
        assert not T.diff_arrays(T.all_results(wb, len(wo), loc), T.all_results(gb, len(go), loc), "batch")
        assert np.array_equal(gb.bundle_counts(), wb.bundle_counts())
        assert len(gs) == len(ws)
        for a, b in zip(gs, ws):
            assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    got.free()
    want.free()
    ctx.close()


def test_two_ranks_paired_gloo(emu_lib):
    res = run_gloo(emu_lib, 2, samples=5, templates=12000, max_batch_hits=20000)
    r0 = res[0]
    assert r0["spanning"] > 0, "no cluster has members on both ranks"
    assert r0["bytes_sent"] > 0
    assert max(g["batches"] for g in r0["ranks"]) >= 2, "the cut by cluster on an owner is exercised: %s" % [g["batches"] for g in r0["ranks"]]


@pytest.mark.parametrize("samples", [4, 2])
def test_three_ranks_single_end_gloo(emu_lib, samples):
    """4 samples: ranks hold 2, 1 and 1 of them; 2 samples: rank 2 holds none and still takes part"""
    res = run_gloo(emu_lib, 3, mode=H.SYNTH_SINGLE, samples=samples, templates=8000)
    r0 = res[0]
    assert r0["spanning"] > 0 and r0["bytes_sent"] > 0
    if samples == 2:
        assert r0["ranks"][2]["exchange"]["bundles_sent"] == 0 and r0["ranks"][2]["exchange"]["bundles_received"] > 0


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_input_columns_adopted_on_another_context_gpu():
    """a gathered batch read through its device columns, cloned into torch memory and adopted on a second context, gives the
    same results as the original on every view"""
    import torch
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 20000, samples=3)
    gp = G.default_params(library_type=lt)
    ctx, ctx2 = G.Context(0), G.Context(0)
    parts = batch.split(2)
    srcs = [ctx.upload(p.view(), keepalive=p) for p in parts]
    glob = np.random.default_rng(3).permutation(batch.n_bundles)
    gb = ctx.gather(srcs, T.picks_of(parts, glob))
    cols = gb.input_columns()
    assert all(t.is_cuda for t in cols.values()) and "bundle_strand" not in cols
    assert cols["pos"].dtype == torch.int32 and cols["qid"].dtype == torch.int64 and cols["strand"].dtype == torch.int8
    sel = batch.select(glob)
    assert np.array_equal(cols["pos"].cpu().numpy(), sel.a["pos"]) and np.array_equal(cols["cigar"].cpu().numpy().view(np.uint32), sel.a["cigar"])
    dev = {k: v.clone() for k, v in cols.items()}
    dev["bundle_tid"] = torch.from_numpy(sel.a["bundle_tid"]).cuda()
    dev["bundle_sample"] = torch.from_numpy(sel.a["bundle_sample"]).cuda()
    torch.cuda.current_stream().synchronize()
    b = H.BatchIn()
    b.n_bundles, b.n_hits, b.n_cigar = sel.n_bundles, sel.n_hits, sel.n_cigar
    for k, t in dev.items():
        setattr(b, k, t.data_ptr())
    adopted = ctx2.adopt(b, keepalive=dev)
    again = ctx2.gather([adopted], [(0, k) for k in range(sel.n_bundles)])
    adopted.free()
    for s in srcs:
        s.free()
    gb.bridge_all(gp)
    again.bridge_all(gp)
    hit_off = sel.a["bundle_hit_off"]
    bad = T.diff_arrays(T.all_results(gb, sel.n_bundles, hit_off), T.all_results(again, sel.n_bundles, hit_off), "adopted")
    assert not bad, bad[:5]
    assert np.array_equal(gb.bundle_counts(), again.bundle_counts())
    gb.free()
    again.free()
    ctx.close()
    ctx2.close()


def _torchrun(args, timeout=1200):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port())] + args
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def _two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")


@pytest.mark.gpu
def test_two_ranks_nccl(tmp_path):
    _two_gpus()
    out = str(tmp_path / "shard.json")
    p = _torchrun([os.path.join(ROOT, "tests", "shard_cluster_worker.py"), "nccl", out, "8", "40000"])
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    r = json.load(open(out))
    assert r["backend"] == "nccl" and r["world"] == 2 and r["spanning"] > 0 and r["bytes_sent"] > 0


@pytest.mark.gpu
def test_cli_two_ranks_equals_one_process(tmp_path):
    _two_gpus()
    cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, seed=20261021)
    s = H.Synth(cfg)
    paths = []
    for k in range(4):
        paths.append(str(tmp_path / ("s%d.bam" % k)))
        H.write_bam(paths[-1], s.sample(k, 15000, threads=4), np.array([cfg.chrom_len], np.int32))
    env = dict(os.environ, PYTHONPATH=ROOT)
    one = subprocess.run([sys.executable, "-m", "aletsch_b200.run", "--clusters"] + paths, capture_output=True, text=True, timeout=900,
                         cwd=ROOT, env=env)
    assert one.returncode == 0, one.stderr[-4000:]
    two = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", str(_free_port()), "-m", "aletsch_b200.run", "--clusters"] + paths,
                         capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert two.returncode == 0, two.stdout[-2000:] + two.stderr[-4000:]
    a = json.loads(one.stdout.strip().splitlines()[-1])
    b = json.loads(two.stdout.strip().splitlines()[-1])
    assert b["ranks"] == 2 and b["clusters_of_bundles"] > 0 and sorted(a) == sorted(b)
    for k in a:
        if k.endswith("_s") or k in ("device_batches", "ranks"):
            continue
        assert a[k] == b[k], "%s: %r (one process) vs %r (two ranks)" % (k, a[k], b[k])
