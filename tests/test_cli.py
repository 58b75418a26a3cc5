"""The command line (aletsch_b200/run.py) on the kernel-logic build: a job that fits one device batch and the same job cut into
several print the same totals, with and without --clusters."""
import json

import numpy as np
import pytest

from aletsch_b200 import clusters as CL
from aletsch_b200 import hostlib as H
from aletsch_b200 import run


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    cfg = H.default_config(H.SYNTH_PAIRED, chrom_len=2_000_000, seed=20261021)
    s = H.Synth(cfg)
    paths = []
    for k in range(3):
        paths.append(str(tmp_path_factory.mktemp("bams") / ("s%d.bam" % k)))
        H.write_bam(paths[-1], s.sample(k, 8000, threads=4), np.array([cfg.chrom_len], np.int32))
    return paths


def _cli(args, capsys):
    assert run.main(args) == 0
    return json.loads(capsys.readouterr().out.strip().splitlines()[-1])


@pytest.mark.parametrize("clusters", [False, True])
def test_cut_job_prints_the_one_batch_totals(emu_lib, bams, clusters, monkeypatch, capsys):
    monkeypatch.setenv("ALETSCH_GPU_LIB", emu_lib)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    args = (["--clusters"] if clusters else []) + bams
    one = _cli(args, capsys)
    monkeypatch.setattr(CL, "MAX_BATCH_HITS", one["hits"] // 4)
    cut = _cli(args, capsys)
    assert one["device_batches"] == 1 and cut["device_batches"] >= 3, (one["device_batches"], cut["device_batches"])
    assert sorted(one) == sorted(cut)
    assert ("region_groups" in one) == clusters and ("clusters_of_bundles" in one) == clusters
    if clusters:
        assert one["region_groups"] > 0 and one["clusters_of_bundles"] > 0
    assert one["bundles"] > 0 and one["bridged"] > 0 and one["ranks"] == 1
    for k in one:
        if not k.endswith("_s") and k != "device_batches":
            assert one[k] == cut[k], "%s: %r (one device batch) vs %r (%d device batches)" % (k, one[k], cut[k], cut["device_batches"])
