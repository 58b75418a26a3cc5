"""SURVEY 8f-4: previewer::infer_insertsize (meta/previewer.cc:151-304) on the C ABI against the reference's own previewer run over
the same records through the htslib stand-in (oracle/ref_driver.cc: ref_infer_insertsize) -- its record loop, its bundle_base with
the never-flushed interval buffer (rnacore/bundle_base.cc:106-204), build_fragments, graph_builder, graph_cluster, the histogram,
the break at max_preview_reads and the percentiles.  CPU tier: kernel-logic build; -m gpu: the CUDA path.  Without the reference
build CASES are compared with the profiles in tests/golden/preview_insertsize.json; its `generated_by` says where they come
from.  `PYTHONPATH=. python tests/test_preview_insertsize.py` rewrites the file from the reference build and fails without it."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import orclib
import parity
from aletsch_b200 import gpu as G, hostlib as H, preview


class RecordsIn(C.Structure):
    _fields_ = [("n", C.c_int64), ("n_chrom", C.c_int32), ("chrom_len", C.c_void_p)] + \
        [(k, C.c_void_p) for k in ("tid", "pos", "mpos", "isize", "flag", "mapq", "xs", "qid", "cigar_off", "cigar")]


def reference_profile(chk, sample, n_chrom, chrom_len, op, max_reads, min_reads, min_hits):
    L = chk.lib
    L.ref_infer_insertsize.argtypes = [C.POINTER(RecordsIn), C.POINTER(orclib.Params), C.c_int, C.c_int, C.c_int, C.c_void_p]
    L.orc_bag_new.restype = C.c_void_p
    r = RecordsIn()
    r.n, r.n_chrom = sample["n"], n_chrom
    cl = np.full(n_chrom, chrom_len, np.int32)
    r.chrom_len = cl.ctypes.data
    keep = [cl]
    for k in ("tid", "pos", "mpos", "isize", "flag", "mapq", "xs", "qid", "cigar_off", "cigar"):
        a = np.ascontiguousarray(sample[k])
        keep.append(a)
        setattr(r, k, a.ctypes.data)
    bag = L.orc_bag_new()
    L.ref_infer_insertsize(C.byref(r), C.byref(op), max_reads, min_reads, min_hits, bag)
    d = chk.bag_to_dict(bag)
    L.orc_bag_free(bag)
    return d


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "preview_insertsize.json")


def stored_profiles():
    """the stored profile of every case of CASES, in reference_profile's layout"""
    with open(GOLDEN) as f:
        g = json.load(f)
    return [{"isize": np.array(d["isize"], np.int32), "isize_d": np.array(d["isize_d"], np.float64)} for d in g["cases"]]


CASES = [(H.FR_FIRST, 1, 40000, 2000000, 100), (H.FR_FIRST, 3, 40000, 2000000, 100), (H.UNSTRANDED, 1, 40000, 2000000, 100),
         (H.UNSTRANDED, 3, 30000, 2000000, 100), (H.FR_SECOND, 2, 30000, 2000000, 100),
         (H.FR_FIRST, 2, 40000, 3000, 100),          # the break at max_preview_reads binds
         (H.FR_FIRST, 1, 2000, 2000000, 100000)]     # fewer fragments than min_preview_spliced_reads: no profile


def run_cases(ctx, chk=None):
    """chk: the reference build's checker, or None to compare with the stored profiles"""
    stored = None if chk is not None else stored_profiles()
    seen_skip = seen_extra = 0
    for i, (lt, n_chrom, templates, max_reads, min_reads) in enumerate(CASES):
        cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, n_chrom=n_chrom, seed=20260500 + 7 * n_chrom + lt)
        s = H.Synth(cfg).sample(0, templates, threads=4)
        gp, op = parity.params_pair(lt)
        pp = H.default_packer_params(lt)
        got = preview.infer_insertsize(ctx, s, pp, gp, max_preview_reads=max_reads, min_preview_spliced_reads=min_reads)
        want = reference_profile(chk, s, n_chrom, 2_000_000, op, max_reads, min_reads, 10) if chk is not None else stored[i]
        where = (lt, n_chrom, templates, max_reads, min_reads)
        assert got["insert_total"] == int(want["isize"][0]), where
        if got["insert_total"] >= min_reads:
            assert [got["insertsize_low"], got["insertsize_high"], got["insertsize_median"]] == want["isize"][1:4].tolist(), where
            assert abs(got["insertsize_ave"] - want["isize_d"][0]) <= parity.REL_TOL * abs(want["isize_d"][0]), where
            assert abs(got["insertsize_std"] - want["isize_d"][1]) <= parity.REL_TOL * abs(want["isize_d"][1]), where
        else:
            assert got["insertsize_low"] is None
        _, _, skip, extra = H.preview_pack(s, pp)
        seen_skip += int((skip != 0).sum())
        seen_extra += len(extra[0])
    assert seen_skip > 0          # the interval-buffer quirk is exercised: blocks without coverage ...
    return seen_extra


def test_preview_insertsize_matches_reference(emu_lib, checkers):
    ctx = G.Context(0, lib_path=emu_lib)
    run_cases(ctx, checkers.get("ref"))
    ctx.close()


def test_interval_buffer_quirk_matters(emu_lib, checkers):
    """the same run WITHOUT the coverage edits is what a clean implementation would compute; the reference's result differs from it
    on at least one of these inputs, i.e. the quirk is observable and the edits are what reproduces it.  Without the reference
    build only the second half is checked."""
    ctx = G.Context(0, lib_path=emu_lib)
    differ = 0
    for seed in range(6):
        cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=1_000_000, n_chrom=2, seed=20260600 + seed)
        s = H.Synth(cfg).sample(0, 30000, threads=4)
        gp, op = parity.params_pair(H.FR_FIRST)
        pp = H.default_packer_params(H.FR_FIRST)
        batch, event, skip, extra = H.preview_pack(s, pp)
        res = []
        for edit in (True, False):
            bt = ctx.upload(batch.view(), keepalive=batch)
            if edit:
                bt.coverage_edit(skip, extra)
            clu_off, isize = bt.preview(gp)
            bt.free()
            res.append((H.insertsize_profile(clu_off, isize, event), isize))
        if "ref" in checkers:
            want = reference_profile(checkers["ref"], s, 2, 1_000_000, op, 2000000, 100, 10)
            assert res[0][0]["insert_total"] == int(want["isize"][0]), seed
        differ += int(len(res[0][1]) != len(res[1][1]) or not np.array_equal(res[0][1], res[1][1]))
    ctx.close()
    assert differ >= 1          # the dropped blocks change graphs / clusters on this data: the quirk is observable


@pytest.mark.gpu
def test_preview_insertsize_matches_reference_gpu(checkers):
    ctx = G.Context(0)
    run_cases(ctx, checkers.get("ref"))
    ctx.close()


def write_golden():
    """record GOLDEN from the reference build's previewer (oracle/_ref); there is no other source"""
    ref = orclib.Checker("ref")
    cases = []
    for lt, n_chrom, templates, max_reads, min_reads in CASES:
        cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, n_chrom=n_chrom, seed=20260500 + 7 * n_chrom + lt)
        s = H.Synth(cfg).sample(0, templates, threads=4)
        _, op = parity.params_pair(lt)
        d = reference_profile(ref, s, n_chrom, 2_000_000, op, max_reads, min_reads, 10)
        cases.append({"isize": [int(x) for x in d["isize"]], "isize_d": [float(x) for x in d["isize_d"]]})
    with open(GOLDEN, "w") as f:
        json.dump({"generated_by": "oracle/_ref/libaletsch_ref.so: ref_infer_insertsize, the reference's previewer", "cases": cases}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":          # from the repository root: PYTHONPATH=. python tests/test_preview_insertsize.py
    write_golden()
