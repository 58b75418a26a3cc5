"""CPU tier, world_size 2 over gloo: the multi-rank plumbing of the path (aletsch_b200/shard.py).
Stages 1-4 shard by bundle with no collective, so the sharded result must equal the single-process result
bundle by bundle; stage 5 all-gathers the splice signatures and must give every rank the single-process groups."""
import os
import socket
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMPLES = 4
TEMPLATES = 12000


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _batch():
    import parity
    from aletsch_b200 import hostlib as H
    return parity.make_batch(H.SYNTH_PAIRED, TEMPLATES, samples=SAMPLES, chrom_len=1_000_000)


def _splice_lists(ctx, batch, gp, bundles):
    """stage 1 on a subset of the bundles (one rank's share), returns their sorted splice lists"""
    from aletsch_b200 import hostlib as H
    sub = batch.select([int(k) for k in bundles])
    bt = ctx.upload(sub.view(), keepalive=sub)
    bt.evidence(gp)
    ev = bt.fetch_evidence(sub.a["bundle_hit_off"])
    cnt = bt.counts()
    bt.free()
    return [e["splices"] for e in ev], [e["seg"] for e in ev], cnt["hits"]


def _worker(rank, world, port, emu, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    import parity
    from aletsch_b200 import gpu as G, shard
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    batch, lt = _batch()
    gp, _ = parity.params_pair(lt, max_group_size=3)
    sizes = np.diff(batch.a["bundle_hit_off"])
    mine = np.nonzero(shard.assign_units(sizes, world) == rank)[0]
    ctx = G.Context(0, lib_path=emu)
    lists, segs, hits = _splice_lists(ctx, batch, gp, mine)
    # one region group of all bundles, keyed by their global indices: clusters in gvv order, members in key order
    off = np.concatenate([[0], np.cumsum([len(x) for x in lists])])
    keys, _, cl_of, owner, _ = shard.resolve_region_groups(ctx, off, np.concatenate(lists), mine, np.zeros(len(mine), np.int64), gp)
    groups = [[(int(owner[i]), int(keys[i])) for i in np.nonzero(cl_of == c)[0]] for c in range(int(cl_of.max()) + 1)]
    ctx.close()
    q.put((rank, mine.tolist(), [x.tolist() for x in lists], [x.tolist() for x in segs], int(hits), groups))
    dist.barrier()
    dist.destroy_process_group()


def test_lpt_assignment_is_balanced_and_total():
    from aletsch_b200 import shard
    rng = np.random.default_rng(7)
    w = rng.integers(1, 100000, 500)
    for world in (1, 2, 4, 8):
        r = shard.assign_units(w, world)
        assert r.min() >= 0 and r.max() < world and len(r) == len(w)
        load = np.array([w[r == k].sum() for k in range(world)])
        assert load.sum() == w.sum()
        assert load.max() - load.min() <= w.max()          # LPT bound
    assert shard.assign_units([], 4).shape == (0,)
    assert list(shard.assign_units([5, 5, 5], 2)) == [0, 1, 0]


def test_two_ranks_resolve_region_groups_match_single_process(emu_lib):
    world = 2
    port = _free_port()
    ctxm = mp.get_context("spawn")
    q = ctxm.Queue()
    procs = [ctxm.Process(target=_worker, args=(r, world, port, emu_lib, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    res.sort()
    # single process over all bundles
    import parity
    from aletsch_b200 import gpu as G
    batch, lt = _batch()
    gp, _ = parity.params_pair(lt, max_group_size=3)
    ctx = G.Context(0, lib_path=emu_lib)
    all_lists, all_segs, all_hits = _splice_lists(ctx, batch, gp, np.arange(batch.n_bundles))
    want_groups = G.group_resolve(ctx, all_lists, gp)
    ctx.close()
    seen = set()
    for rank, mine, lists, segs, hits, groups in res:
        for k, l, s in zip(mine, lists, segs):
            assert l == all_lists[k].tolist() and s == all_segs[k].tolist(), "bundle %d differs when sharded" % k
            seen.add(k)
    assert seen == set(range(batch.n_bundles))
    assert sum(r[4] for r in res) == all_hits
    # every rank resolved the same groups, equal to the single-process ones (keys are the global bundle indices)
    g0 = [[k for _, k in g] for g in res[0][5]]
    g1 = [[k for _, k in g] for g in res[1][5]]
    assert g0 == g1 == want_groups
    assert max(len(g) for g in want_groups) == 3          # the size cap binds
    owners = {k: r for g in res[0][5] for r, k in g}
    for rank, mine, *_ in res:
        assert all(owners[k] == rank for k in mine)
