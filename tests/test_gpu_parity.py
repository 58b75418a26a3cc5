"""-m gpu: parity of the CUDA path (through the C ABI) against the CPU checkers on a B200."""
import numpy as np
import pytest

import parity
from aletsch_b200 import gpu as G
from aletsch_b200 import hostlib as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = G.Context(0)          # raises if libaletsch_gpu.so is missing or no device: no CPU fallback
    yield c
    c.close()


@pytest.mark.parametrize("mode,templates", [(H.SYNTH_PAIRED, 30000), (H.SYNTH_SINGLE, 20000), (H.SYNTH_LONG, 3000)])
def test_evidence_graph_parity(ctx, checkers, mode, templates):
    assert checkers, "no CPU checker library found (oracle/liboracle.so or oracle/_ref/libaletsch_ref.so)"
    batch, lt = parity.make_batch(mode, templates)
    assert batch.n_bundles > 0
    gp, op = parity.params_pair(lt)
    for name, chk in checkers.items():
        bad = parity.compare_evidence_graph(ctx, batch, chk, gp, op)
        assert not bad, "%s: %d mismatches, first: %s" % (name, len(bad), bad[:3])


@pytest.mark.parametrize("mode,templates,seed", [(H.SYNTH_PAIRED, 60000, 20260101), (H.SYNTH_PAIRED, 150000, 20260102),
                                                 (H.SYNTH_SINGLE, 20000, 20260104), (H.SYNTH_LONG, 3000, 20260105)])
def test_bundle_bridge_parity(ctx, checkers, mode, templates, seed):
    """the whole per-bundle path (bundle::bridge) with every intermediate compared"""
    assert checkers
    batch, lt = parity.make_batch(mode, templates, seed=seed)
    gp, op = parity.params_pair(lt)
    for name, chk in checkers.items():
        stats = {}
        bad = parity.compare_full(ctx, batch, chk, gp, op, stats)
        assert not bad, "%s: %d mismatches, first: %s" % (name, len(bad), bad[:3])
        if mode == H.SYNTH_PAIRED:
            assert stats["bridged"] > 0 and stats["clusters"] > 0


@pytest.mark.parametrize("first_round", [True, False])
def test_group_bridge_parity(ctx, checkers, first_round):
    """assembler::bridge: clusters of bundles merged into combined bundles (chain sets, coverage maps, bounds), the combined
    splice graph, and every member re-clustered / re-bridged / updated against it"""
    assert checkers
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 30000, samples=4)
    gp, op = parity.params_pair(lt)
    groups = parity.locus_groups(batch)
    assert len(groups) >= 4
    for name, chk in checkers.items():
        stats = {}
        bad = parity.compare_group_bridge(ctx, batch, chk, gp, op, groups, stats, first_round=first_round)
        assert not bad, "%s: %d mismatches, first: %s" % (name, len(bad), bad[:3])
        assert stats["group_bridged"] == stats["ref_group_bridged"]
        if not first_round:
            assert stats["group_bridged"] > 0


@pytest.mark.parametrize("mode,templates,samples", [(H.SYNTH_PAIRED, 60000, 4), (H.SYNTH_PAIRED, 60000, 6), (H.SYNTH_SINGLE, 30000, 4)])
def test_group_support_parity(ctx, checkers, mode, templates, samples):
    """the cross-sample support features of assembler::assemble(vector<bundle*>) (meta/assembler.cc:177-373): junction_support,
    start_end_support, non_splicing_support and boundary_extend over the members' revised graphs and the combined graph, with the
    boundary regrouping of the members already assembled -- against the reference's own functions driven in its order (scallop
    left out) and against the restatement"""
    assert checkers
    batch, lt = parity.make_batch(mode, templates, samples=samples)
    gp, op = parity.params_pair(lt)
    groups = parity.locus_groups(batch, max_groups=30)
    assert len(groups) >= 5
    for name, chk in checkers.items():
        stats = {}
        bad = parity.compare_group_support(ctx, batch, chk, gp, op, groups, stats)
        assert not bad, "%s: %d mismatches, first: %s" % (name, len(bad), bad[:3])
        assert stats["support_edges"] > 100 and stats["support_multi"] > 0


@pytest.mark.parametrize("mode,templates", [(H.SYNTH_PAIRED, 40000), (H.SYNTH_SINGLE, 20000), (H.SYNTH_LONG, 3000)])
def test_phase_set_parity(ctx, checkers, mode, templates):
    """build_phase_set: phasing paths of bridged fragments and unpaired hits, counted and in phase_set::pmap order"""
    assert checkers
    batch, lt = parity.make_batch(mode, templates)
    gp, op = parity.params_pair(lt)
    for name, chk in checkers.items():
        stats = {}
        bad = parity.compare_phase_set(ctx, batch, chk, gp, op, stats)
        assert not bad, "%s: %d mismatches, first: %s" % (name, len(bad), bad[:3])
        assert stats["phase_count"] > 0


@pytest.mark.parametrize("mode,templates", [(H.SYNTH_PAIRED, 40000), (H.SYNTH_SINGLE, 20000), (H.SYNTH_LONG, 3000)])
def test_revise_parity(ctx, checkers, mode, templates):
    """identify_boundaries + remove_false_boundaries: added boundary edges in order, the revised graph, vertex annotations"""
    assert checkers
    batch, lt = parity.make_batch(mode, templates)
    # 2.0 is the reference's default (few runs qualify in the synthetic transcriptome); lower thresholds make the rounds long
    for ratio in (2.0, 1.1, 0.6):
        gp, op = parity.params_pair(lt, min_boundary_log_ratio=ratio)
        for name, chk in checkers.items():
            stats = {}
            bad = parity.compare_revise(ctx, batch, chk, gp, op, stats)
            assert not bad, "%s ratio %.1f: %d mismatches, first: %s" % (name, ratio, len(bad), bad[:3])
            assert ratio > 1.5 or stats["rev_added"] > 10
            if mode == H.SYNTH_PAIRED:
                assert stats["rev_marked"] > 0


@pytest.mark.parametrize("mode,templates", [(H.SYNTH_PAIRED, 60000), (H.SYNTH_SINGLE, 20000), (H.SYNTH_LONG, 3000)])
def test_reference_scallop_on_adapter_graphs(ctx, checkers, mode, templates):
    """the reference's own assembler + scallop fed from the C-ABI views through integration/adapter.cc: rebuilt graph / phase
    set equal to the reference's field by field; identical transcripts wherever the reference agrees with itself"""
    import test_adapter_transcripts as T
    T.run_case(ctx, checkers, mode, templates)


@pytest.mark.parametrize("mode,templates", [(H.SYNTH_PAIRED, 30000), (H.SYNTH_LONG, 3000)])
def test_compact_upload_matches_full(ctx, mode, templates):
    """agpu_batch_upload_packed: 16-bit deltas / offsets / CIGAR units with escapes, decoded on the device"""
    batch, lt = parity.make_batch(mode, templates)
    stats = {}
    bad = parity.compare_compact_upload(ctx, batch, G.default_params(library_type=lt), stats)
    assert not bad, bad[:3]
    assert stats["bytes_compact"] < 0.75 * stats["bytes_full"], stats
    assert stats["long_ops"] > 0, stats
    assert mode != H.SYNTH_PAIRED or stats["default_cigars"] > batch.n_hits // 4, stats


def test_compact_upload_escapes_and_errors(ctx):
    """values that do not fit 16 bits travel through the escape lists; a sentinel without its entry is an input error"""
    import fuzz
    batch = fuzz.random_batch(5, n_bundles=6, max_hits=80)
    a = batch.a
    rng = np.random.default_rng(5)
    far = rng.choice(batch.n_hits, 12, replace=False)
    a["mpos"][far[:6]] += 70000                      # mate far away
    a["isize"][far[6:]] = 40000 + np.arange(6, dtype=np.int32)
    # a jump of more than 65534 bases inside a bundle: shift the tail of the largest bundle
    k = int(np.argmax(np.diff(a["bundle_hit_off"])))
    h0, h1 = int(a["bundle_hit_off"][k]), int(a["bundle_hit_off"][k + 1])
    mid = (h0 + h1) // 2
    for f in ("pos", "rpos", "mpos"):
        a[f][mid:h1] += 100000
    gp = G.default_params(library_type=H.FR_FIRST)
    stats = {}
    bad = parity.compare_compact_upload(ctx, batch, gp, stats)
    assert not bad, bad[:3]
    assert stats["escapes"] >= 13, stats
    arrays = batch.compact()
    arrays["esc_isize_idx"] = arrays["esc_isize_idx"][:-1].copy()          # drop an entry a sentinel points to
    arrays["esc_isize_val"] = arrays["esc_isize_val"][:-1].copy()
    with pytest.raises(G.AgpuError) as e:
        ctx.upload(H.compact_struct(arrays, batch.n_cigar), keepalive=(arrays, batch))
    assert "escape entry" in str(e.value) and "-4" in str(e.value)          # AGPU_ERR_INPUT


def test_device_path_matches_committed_fixtures(ctx):
    """no checker library in the loop: the fixtures under tests/golden were written by the reference build"""
    import os
    bad, n = parity.compare_golden(ctx, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    assert not bad, bad[:3]
    assert n > 300


def test_lean_upload_matches_full(ctx):
    """rpos / flag / per-hit strand are optional in agpu_batch_in (include/aletsch_gpu.h)"""
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 20000)
    gp, _ = parity.params_pair(lt)
    bad = parity.compare_lean_upload(ctx, batch, gp)
    assert not bad, bad[:3]


def test_group_resolve_parity(ctx, checkers):
    """bundle_group::resolve: device similarity + host control flow against the checker, with the size cap binding"""
    import numpy as np
    from aletsch_b200 import gpu as G
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 30000, samples=6)
    gp, op = parity.params_pair(lt, max_group_size=4)
    n = min(batch.n_bundles, 200)
    for name, chk in checkers.items():
        hs = [chk.new_bundle(batch.bundle(k), op) for k in range(n)]
        lists = [chk.run(h, "evidence")[1]["splices"] for h in hs]
        _, gr = chk.group_resolve(hs, op)
        for h in hs:
            chk.free_bundle(h)
        want = [gr["gvv_val"][gr["gvv_off"][i]:gr["gvv_off"][i + 1]].tolist() for i in range(len(gr["gvv_off"]) - 1)]
        got = G.group_resolve(ctx, lists, gp)
        assert got == want, name
        assert max(len(g) for g in want) == 4
    c, r = ctx.similarity(lists)
    for i in range(0, n, 7):
        for j in range(i + 1, n, 3):
            cc = len(np.intersect1d(lists[i], lists[j]))
            assert cc == c[i, j]
            if cc:
                assert abs(r[i, j] - cc / min(len(lists[i]), len(lists[j]))) <= 1e-9 * r[i, j]       # BASELINE.json tolerance


def test_group_resolve_batch_matches_single(ctx):
    """many bundle groups in one call (one CTA per group) == one call per group; includes an empty group, a singleton and a
    group above the one-CTA limit"""
    import numpy as np
    rng = np.random.default_rng(11)
    groups = []
    for gsize in (0, 1, 2, 7, 40, 200, 13):
        pool = np.sort(rng.choice(200000, size=60, replace=False)).astype(np.int32)
        grp = []
        for _ in range(gsize):
            k = int(rng.integers(0, 12)) * 2
            grp.append(np.sort(rng.choice(pool, size=k, replace=False)).astype(np.int32))
        groups.append(grp)
    gp = G.default_params(max_group_size=5, min_grouping_similarity=0.2)
    got = G.group_resolve_batch(ctx, groups, gp)
    for grp, g in zip(groups, got):
        want = G.group_resolve(ctx, grp, gp) if len(grp) else []
        assert g == want


def test_fuzz_bundles(ctx, checkers):
    """adversarial random bundles (tests/fuzz.py), small and large (big qname / cluster groups reach the warp kernels)"""
    import test_fuzz
    test_fuzz.run_seeds(ctx, checkers, range(24))
    test_fuzz.run_seeds(ctx, checkers, range(100, 104), big=True)
    test_fuzz.run_degenerate(ctx, checkers)
    test_fuzz.run_group_seeds(ctx, checkers, range(16))
    test_fuzz.run_pair_seeds(ctx, checkers, range(12))


CHILD_PRELUDE = ("import sys; sys.path.insert(0, 'tests'); import parity, orclib, test_fuzz\n"
                 "from aletsch_b200 import gpu as G, hostlib as H\n"
                 "checkers = {}\n"
                 "for p in ('ref', 'orc'):\n"
                 "    try:\n"
                 "        checkers[p] = orclib.Checker(p)\n"
                 "    except (OSError, FileNotFoundError):\n"
                 "        pass\n"
                 "assert checkers\n"
                 "chk = checkers.get('ref') or next(iter(checkers.values()))\n"
                 "ctx = G.Context(0)\n")


def run_child(env, body, marker):
    """a parity run in a child process: the library reads its path switches from the environment once per process"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", CHILD_PRELUDE + body], cwd=root, env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert marker in r.stdout


def test_pairing_exact_path_at_scale():
    """AGPU_PAIR_EXACT=1 sends EVERY hit that has a mate candidate through the exact per-(bundle, qname) greedy (the path only
    multi-mapped query names take otherwise): same fragments as the reference on a batch of 60,000 templates."""
    run_child({"AGPU_PAIR_EXACT": "1"},
              "batch, lt = parity.make_batch(H.SYNTH_PAIRED, 60000, seed=20260111)\n"
              "gp, op = parity.params_pair(lt)\n"
              "stats = {}; bad = parity.compare_full(ctx, batch, chk, gp, op, stats)\n"
              "assert not bad, bad[:3]\n"
              "assert stats['fragments'] > 10000\n"
              "print('exact path ok', stats['fragments'])\n", "exact path ok")


def test_pairing_long_runs_take_exact_path():
    """AGPU_PAIR_RUN_MAX=2: a bundle in which some mate position holds more than two hits goes through the exact greedy as a
    whole (the bound that keeps R reads at one start position from costing R^2 candidate walks; 1024 by default)."""
    run_child({"AGPU_PAIR_RUN_MAX": "2"},
              "test_fuzz.run_pair_seeds(ctx, checkers, range(6))\n"
              "test_fuzz.run_seeds(ctx, checkers, range(6))\n"
              "batch, lt = parity.make_batch(H.SYNTH_PAIRED, 60000, seed=20260113)\n"
              "gp, op = parity.params_pair(lt)\n"
              "stats = {}; bad = parity.compare_full(ctx, batch, chk, gp, op, stats)\n"
              "assert not bad, bad[:3]\n"
              "print('long runs ok', stats['fragments'])\n", "long runs ok")


def test_warp_cigar_walk_on_short_reads():
    """AGPU_WARP_MIN_OPS=0 runs the warp-per-hit CIGAR walks (the long-read path: k_hit_cigar_warp, k_cov_add_warp,
    k_hit_rpos_warp) on every batch: adversarial CIGARs of 1-9 operations, the synthetic paired-end batch through the compact
    upload (rpos derived on the device), and the insert-size preview (the skip mask of the match blocks)."""
    run_child({"AGPU_WARP_MIN_OPS": "0"},
              "test_fuzz.run_seeds(ctx, checkers, range(10))\n"
              "test_fuzz.run_seeds(ctx, checkers, range(100, 102), big=True)\n"
              "batch, lt = parity.make_batch(H.SYNTH_PAIRED, 30000, seed=20260112)\n"
              "gp, op = parity.params_pair(lt)\n"
              "stats = {}; bad = parity.compare_full(ctx, batch, chk, gp, op, stats)\n"
              "assert not bad, bad[:3]\n"
              "import test_gpu_parity as T\n"
              "T.test_compact_upload_matches_full(ctx, H.SYNTH_PAIRED, 20000)\n"
              "import test_preview_insertsize as P\n"
              "P.run_cases(ctx, checkers.get('ref'))\n"
              "print('warp walk ok', stats['segments'])\n", "warp walk ok")


def test_long_read_scale_parity(ctx, checkers):
    """configs[4]-style input at a larger scale: many-junction long reads (junction / coverage-heavy path), ONT junction support"""
    batch, lt = parity.make_batch(H.SYNTH_LONG, 20000, chrom_len=4_000_000, seed=20260105)
    gp, op = parity.params_pair(lt, min_junction_support=2)
    chk = checkers.get("ref") or next(iter(checkers.values()))
    stats = {}
    bad = parity.compare_full(ctx, batch, chk, gp, op, stats)
    assert not bad, bad[:3]
    assert stats["junctions"] > 100


def test_bam_file_to_device(ctx, tmp_path):
    """BAM file -> host ingest -> packer -> CUDA path (python -m aletsch_b200.run does the same): identical to the direct path"""
    import numpy as np
    cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=1_000_000, seed=20260113)
    syn = H.Synth(cfg)
    recs = [syn.sample(k, 8000, threads=2) for k in range(2)]
    back = []
    for k, r in enumerate(recs):
        path = str(tmp_path / ("s%d.bam" % k))
        H.write_bam(path, r, [cfg.chrom_len] * cfg.n_chrom)
        back.append(H.read_bam(path)[0])
    pp = H.default_packer_params(H.FR_FIRST)
    gp, _ = parity.params_pair(H.FR_FIRST)
    outs = []
    for b in (H.pack(recs, pp), H.pack(back, pp)):
        bt = ctx.upload(b.view(), keepalive=b)
        bt.bridge_all(gp)
        outs.append((bt.counts(), bt.bundle_counts().copy()))
        bt.free()
    assert outs[0][0] == outs[1][0] and np.array_equal(outs[0][1], outs[1][1]) and outs[0][0]["bridged"] > 0


def test_single_cell_group_resolve(ctx, checkers):
    """configs[3]-style input: many cells, each expressing a fraction of the genes, clustered with a large -c: one bundle group
    of many hundred small graphs (beyond the one-CTA limit of the batched kernel -> the tiled AND-popcount kernels)"""
    batch, lt = parity.make_batch(H.SYNTH_SINGLE, 1200, samples=500, chrom_len=400_000, expressed_fraction=0.3)
    gp, op = parity.params_pair(lt, max_group_size=2000, min_grouping_similarity=0.2)
    chk = checkers.get("ref") or next(iter(checkers.values()))
    hs = [chk.new_bundle(batch.bundle(k), op) for k in range(batch.n_bundles)]
    lists = [chk.run(h, "evidence")[1]["splices"] for h in hs]
    _, gr = chk.group_resolve(hs, op)
    for h in hs:
        chk.free_bundle(h)
    want = [gr["gvv_val"][gr["gvv_off"][i]:gr["gvv_off"][i + 1]].tolist() for i in range(len(gr["gvv_off"]) - 1)]
    assert batch.n_bundles > 700
    assert G.group_resolve(ctx, lists, gp) == want
    assert G.group_resolve_batch(ctx, [lists], gp)[0] == want
    assert max(len(g) for g in want) > 20


def test_packing_contract_violations_are_reported(ctx):
    """agpu_batch_evidence verifies the packing contract of agpu_batch_in on the device and returns AGPU_ERR_INPUT (-4)"""
    import numpy as np
    import fuzz
    gp, _ = parity.params_pair(H.FR_FIRST)

    def run(mutate, rpos=True):
        b = fuzz.random_batch(5, n_bundles=3, max_hits=30)
        mutate(b.a)
        v = b.view()
        if not rpos:
            v.rpos = None
        bt = ctx.upload(v, keepalive=b)
        try:
            bt.evidence(gp)
        finally:
            bt.free()

    run(lambda a: None)                                                   # the untouched batch is fine
    cases = {"hit order": lambda a: a["pos"].__setitem__(1, a["pos"][0] - 5),
             "duplicate": lambda a: (a["pos"].__setitem__(1, a["pos"][0]), a["rpos"].__setitem__(1, a["rpos"][0]),
                                     a["cigar"].__setitem__(slice(int(a["cigar_off"][1]), int(a["cigar_off"][2])), 0)),
             "strand": lambda a: a["strand"].__setitem__(1, ord("-") if a["strand"][0] == ord("+") else ord("+")),
             "rpos": lambda a: a["rpos"].__setitem__(0, a["rpos"][0] + 1)}
    for name, mut in cases.items():
        with pytest.raises(G.AgpuError) as e:
            run(mut)
        assert "failed with -4" in str(e.value), (name, str(e.value))
    # a wrong rpos cannot happen when the device derives it
    run(cases["rpos"], rpos=False)


def test_huge_bundle_parity(ctx, checkers):
    """two bundles of ~190,000 hits each over overlapping genes (graphs of thousands of vertices, thousands of piers): the wide
    CTA paths of the per-bundle kernels, big qname / cluster groups, long DP jobs"""
    batch, lt = parity.make_batch(H.SYNTH_PAIRED, 500000, chrom_len=1_000_000, seed=5, gene_spacing=1500)
    assert batch.n_bundles <= 4 and batch.n_hits > 300000
    gp, op = parity.params_pair(lt)
    chk = checkers.get("ref") or next(iter(checkers.values()))
    stats = {}
    bad = parity.compare_full(ctx, batch, chk, gp, op, stats)
    assert not bad, bad[:3]
    assert stats["vertices"] > 3000 and stats["piers"] > 3000 and stats["bridged"] > 50000


def test_std_sort_permutation(ctx):
    """the device re-implementation of libstdc++'s introsort against the real std::sort on heavily tied keys"""
    import ctypes as C
    import numpy as np
    import orclib
    L = C.CDLL(orclib.ORC_SO)
    L.orc_std_sort_perm.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    rng = np.random.default_rng(5)
    # 17 .. 32: one element per lane in registers; 33 .. 128: in shared memory; above: the warp-cooperative replay in global memory
    sizes = [1, 2, 15, 16] + list(range(17, 34)) + [47, 48, 49, 64, 65, 100, 127, 128, 129, 257, 1000, 4096, 20000]
    for n in sizes:
        for kind in range(10):
            if kind >= 6:
                keys = rng.integers(0, (2, 3, 8, 1 << 20)[kind - 6], n)
            elif kind == 0:
                keys = rng.integers(0, 4, n)
            elif kind == 1:
                keys = rng.integers(0, max(2, n // 3), n)
            elif kind == 2:
                keys = np.arange(n) // 5
            elif kind == 3:
                keys = (np.arange(n)[::-1]) // 3
            elif kind == 4:
                keys = np.minimum(np.arange(n), np.arange(n)[::-1])          # organ pipe
            else:
                keys = np.zeros(n)
            keys = np.ascontiguousarray(keys, np.int32)
            want = np.zeros(n, np.int32)
            L.orc_std_sort_perm(keys.ctypes.data, n, want.ctypes.data)
            got = ctx.sort_perm(keys)
            assert np.array_equal(got, want), (n, kind)
